"""One grasp-refinement step's nearest-point search at the grasp batch: B = 4096 hands of 778 vertices, objects of 3000
points (4096 * 3000 * 778 = 9.56e9 point pairs per direction), dvq kernels against a plain-torch brute force:

    python scripts/bench_contact.py [--out profiles/r05_bench_contact.json] [--reps 5] [--iters 10]

dvq stages, each timed with CUDA events around --iters calls after warm-up:
  obj_to_hand   dvq.HandObjectContact: vertex normals + object -> hand search with the interior mask (no autograd)
  hand_to_obj   dvq.nearest_points(hand, obj) (no autograd)
  backward      dvq_nn_backward of both directions with respect to the hand vertices (g_trg of the first, g_src of the second)
  total         the sum of the three
The torch arm is what a caller without pytorch3d writes: the float32 broadcast-difference distance tensor, min over the
last axis, and its autograd backward to the hand vertices, both directions, chunked over B to fit memory.  The arms
alternate within each of --reps repetitions; medians are reported.  The working set (185 MB of points) is larger than the
126 MB L2, so every step reads its inputs from HBM.  The two arms' indices are compared: any disagreement must be a
near-tie (float64 distances to both picks within 1e-6 relative).  Prints one JSON line and writes it to --out."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "d-vqvae_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dvq  # noqa: E402
from dvq import _cabi  # noqa: E402
from oracle import mano_oracle as mo  # noqa: E402

B, P, V = 4096, 3000, 778
TIE = 1e-6


def card():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = (x.strip() for x in r.stdout.strip().split(","))
    return name, power, clock


def torch_nn(src, trg):
    """float32 brute force of one chunk: (dist, idx) with autograd through dist"""
    d = ((src[:, :, None, :] - trg[:, None, :, :]) ** 2).sum(-1)
    return d.min(-1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bench_contact.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=256, help="batch items per torch chunk")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_contact.py measures on the GPU"
    dev = torch.device("cuda:0")
    name, power, clock = card()
    model = mo.synthetic_model(0)
    layer = dvq.ManoLayer(model).to(dev)
    contact = dvq.HandObjectContact(layer.faces).to(dev)
    rs = np.random.RandomState(0)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    with torch.no_grad():
        hand = layer(betas=cuda(rs.randn(B, 10)), hand_pose=cuda(0.5 * rs.randn(B, 45)), global_orient=cuda(0.3 * rs.randn(B, 3))).vertices
    centre = hand.mean(1, keepdim=True)
    obj = (centre + 0.04 * cuda(rs.randn(B, P, 3))).contiguous()     # an object cloud around each hand
    pairs = B * P * V

    # dvq backward buffers (the upstream gradients of a mean-reduced loss)
    g1 = torch.full((B, P), 1.0 / (B * P), device=dev)
    g2 = torch.full((B, V), 1.0 / (B * V), device=dev)
    g_hand1, g_hand2 = torch.empty_like(hand), torch.empty_like(hand)
    stream = lambda: torch.cuda.current_stream(dev).cuda_stream
    state = {}

    def obj_to_hand():
        with torch.no_grad():
            state["o2h"] = contact(hand, obj)

    def hand_to_obj():
        with torch.no_grad():
            state["h2o"] = dvq.nearest_points(hand, obj)

    def backward():
        _cabi.check(_cabi.lib.dvq_nn_backward(obj.data_ptr(), hand.data_ptr(), state["o2h"][1].data_ptr(), g1.data_ptr(), B, P, V,
                                              None, g_hand1.data_ptr(), stream()), "dvq_nn_backward")
        _cabi.check(_cabi.lib.dvq_nn_backward(hand.data_ptr(), obj.data_ptr(), state["h2o"][1].data_ptr(), g2.data_ptr(), B, V, P,
                                              g_hand2.data_ptr(), None, stream()), "dvq_nn_backward")

    def torch_step():
        idx = [[], []]
        for b0 in range(0, B, args.chunk):
            h = hand[b0:b0 + args.chunk].detach().requires_grad_(True)
            o = obj[b0:b0 + args.chunk]
            d1, i1 = torch_nn(o, h)
            d2, i2 = torch_nn(h, o)
            (d1.sum() / (B * P) + d2.sum() / (B * V)).backward()
            idx[0].append(i1)
            idx[1].append(i2)
        state["torch_idx"] = [torch.cat(i) for i in idx]

    stages = {"obj_to_hand": obj_to_hand, "hand_to_obj": hand_to_obj, "backward": backward}
    for _ in range(args.warmup):
        for f in stages.values():
            f()
    torch_step()
    torch.cuda.synchronize()

    def timed(f, iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            f()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / iters

    times = {k: [] for k in list(stages) + ["torch_step"]}
    for _ in range(args.reps):
        for k, f in stages.items():
            times[k].append(timed(f, args.iters))
        times["torch_step"].append(timed(torch_step, 1))
    med = {k: statistics.median(t) for k, t in times.items()}
    total = med["obj_to_hand"] + med["hand_to_obj"] + med["backward"]

    # index agreement between the arms (outside the near-tie band)
    agree = {}
    for name_, (src, trg, ours, theirs) in {"obj_to_hand": (obj, hand, state["o2h"][1], state["torch_idx"][0]),
                                            "hand_to_obj": (hand, obj, state["h2o"][1], state["torch_idx"][1])}.items():
        mis = (ours != theirs).nonzero()
        b, i = mis[:, 0], mis[:, 1]
        s = src[b, i].double()
        da = ((s - trg[b, ours[b, i]].double()) ** 2).sum(-1)
        db = ((s - trg[b, theirs[b, i]].double()) ** 2).sum(-1)
        outside = int(((da - db).abs() > TIE * torch.minimum(da, db) + 1e-12).sum())
        agree[name_] = {"rows": int(ours.numel()), "idx_differ": int(mis.shape[0]), "differ_outside_near_tie_band": outside}
    rate = lambda ms: pairs / (ms * 1e-3)
    res = {"card": name, "power_limit": power, "max_sm_clock": clock,
           "workload": "B=%d hands (synthetic MANO model, random pose) x %d hand vertices, %d object points around each hand; "
                       "%.3g point pairs per direction; %.0f MB of points, larger than the 126 MB L2" % (B, V, P, pairs, (hand.numel() + obj.numel()) * 4 / 1e6),
           "method": "CUDA events around %d calls per dvq stage and 1 torch step, after warm-up; the arms alternate within each of %d "
                     "repetitions; medians" % (args.iters, args.reps),
           "dvq": {"obj_to_hand_with_normals_and_interior": {"ms": med["obj_to_hand"], "pairs_per_s": rate(med["obj_to_hand"])},
                   "hand_to_obj": {"ms": med["hand_to_obj"], "pairs_per_s": rate(med["hand_to_obj"])},
                   "backward_both_wrt_hand": {"ms": med["backward"], "pairs_per_s": 2 * rate(med["backward"])},
                   "total": {"ms": total, "pairs_per_s": 2 * rate(total)}},
           "torch_brute_force_fp32": {"forward_backward_both_ms": med["torch_step"], "chunk": args.chunk,
                                      "pairs_per_s": 2 * rate(med["torch_step"])},
           "speedup_total_vs_torch": med["torch_step"] / total,
           "idx_check": agree,
           "ms_all": times}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()

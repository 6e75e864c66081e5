"""Differentiable penetration at the generation batch, on bench_grasp_quality.py's workload: B = 4096 closed hand-sized
ellipsoids (642 vertices / 1280 faces) at random poses around an icosphere object of radius 5 cm (5120 faces), voxel
pitch 5 mm.

    python scripts/bench_penetration.py [--out profiles/r07_bench_penetration.json] [--reps 5] [--iters 5]

CUDA events around --iters calls of each stage after warm-up, medians over --reps repetitions (the stages alternate
within each repetition):
  hand_fused / hand_composed    hand vertices against the object: dvq.penetration_depth, against winding_number +
                                point_mesh_distance + torch.where (the two launches and the select it replaces)
  voxel_fused / voxel_composed  the object's voxel centres (GraspQuality.centres) against every hand, the same two ways
  hand_backward / voxel_backward  dvq_mesh_distance_backward of each direction (g_pts and g_verts)
  refine_step                   one refinement step: ManoLayer(differentiable=True) forward on synthetic tables, both
                                penetration terms forward and backward, the MANO backward
  torch_autograd                a chunked fp32 torch arm on the first --torch-batch hands: the same winding (no grad) and
                                Ericson distances as tensors, torch.where, autograd backward to the hand vertices
The fused and composed outputs are compared bit for bit on the whole batch, and the torch arm's depth2 and gradient
against dvq's on its hands.  Prints one JSON line and writes it to --out."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "d-vqvae_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dvq  # noqa: E402
from bench_grasp_quality import B, PITCH, TOL, card, torch_distance, torch_winding  # noqa: E402
from oracle import mano_oracle as mano  # noqa: E402
from test_contact import icosphere  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_bench_penetration.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--torch-batch", type=int, default=64)
    ap.add_argument("--chunk", type=int, default=2, help="hands per torch chunk")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_penetration.py measures on the GPU"
    dev = torch.device("cuda:0")
    name, power, clock = card()
    rs = np.random.RandomState(0)                                        # bench_grasp_quality.py's hands, same seed
    ov, of = icosphere(0.05, 4)
    hv, hf = icosphere(1.0, 3)
    hv = hv * np.array([0.045, 0.02, 0.012])
    d = rs.randn(B, 3)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rot = np.linalg.qr(rs.randn(B, 3, 3))[0]
    rot *= np.linalg.det(rot)[:, None, None]
    hands_np = np.einsum("vk,bjk->bvj", hv, rot) + (rs.uniform(0.0, 0.1, (B, 1)) * d)[:, None, :]
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    obj, hands = cuda(ov), cuda(hands_np)
    gq = dvq.GraspQuality(obj, of, hf, PITCH, TOL).to(dev)
    O, C = gq.obj_verts, gq.centres
    zero = torch.zeros((), device=dev)

    def composed(q, v, f):
        w = dvq.winding_number(q, v, f)
        d2, face = dvq.point_mesh_distance(q, v, f)
        ins = w >= 0.5
        return torch.where(ins, d2, zero), torch.where(ins, face, torch.full((), -1, device=dev))

    state = {}
    hand_g = hands.clone().requires_grad_(True)
    hd2, _ = dvq.penetration_depth(hand_g, O, of)
    vox_g = hands.clone().requires_grad_(True)
    vd2, _ = dvq.penetration_depth(C, vox_g, hf)
    g_hand, g_vox = torch.ones_like(hd2), torch.ones_like(vd2)

    # refinement: synthetic MANO tables scaled to hand size, hands placed around the object
    model = mano.synthetic_model(3)
    model["v_template"] = 0.3 * model["v_template"]
    layer = dvq.ManoLayer(model, differentiable=True).to(dev)
    mfaces = layer.faces
    params = [cuda(0.3 * rs.randn(B, 10)), cuda(0.3 * rs.randn(B, 3)), cuda(0.3 * rs.randn(B, 45)), cuda(0.05 * rs.randn(B, 3))]
    params = [p.requires_grad_(True) for p in params]

    def refine_step():
        for p in params:
            p.grad = None
        verts = layer(betas=params[0], global_orient=params[1], hand_pose=params[2], transl=params[3]).vertices
        a, _ = dvq.penetration_depth(verts, O, of)
        b, _ = dvq.penetration_depth(C, verts, mfaces)
        ((a.sum() + b.sum()) / B).backward()
        state["refine"] = (a.detach(), b.detach())

    stages = {
        "hand_fused": lambda: state.__setitem__("hand_fused", dvq.penetration_depth(hands, O, of)),
        "hand_composed": lambda: state.__setitem__("hand_composed", composed(hands, O, of)),
        "voxel_fused": lambda: state.__setitem__("voxel_fused", dvq.penetration_depth(C, hands, hf)),
        "voxel_composed": lambda: state.__setitem__("voxel_composed", composed(C, hands, hf)),
        "hand_backward": lambda: torch.autograd.grad(hd2, hand_g, g_hand, retain_graph=True),
        "voxel_backward": lambda: torch.autograd.grad(vd2, vox_g, g_vox, retain_graph=True),
        "refine_step": refine_step,
    }

    T = args.torch_batch
    obj_tri = obj[torch.from_numpy(of).to(dev)][None]
    olo, ohi = obj.min(0).values[None], obj.max(0).values[None]

    def torch_arm():
        d2s, grads = [], []
        for b0 in range(0, T, args.chunk):
            h = hands[b0:min(T, b0 + args.chunk)].clone().requires_grad_(True)
            n = h.shape[0]
            with torch.no_grad():
                ins = torch_winding(h, obj_tri, olo.expand(n, -1), ohi.expand(n, -1)) >= 0.5
            d2 = torch.where(ins, torch_distance(h, obj_tri), zero)
            d2.sum().backward()
            d2s.append(d2.detach())
            grads.append(h.grad)
        state["torch"] = (torch.cat(d2s), torch.cat(grads))

    for _ in range(args.warmup):
        for f in stages.values():
            f()
    torch_arm()
    torch.cuda.synchronize()

    def timed(f, iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            f()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / iters

    times = {k: [] for k in list(stages) + ["torch_autograd"]}
    for _ in range(args.reps):
        for k, f in stages.items():
            times[k].append(timed(f, args.iters))
        times["torch_autograd"].append(timed(torch_arm, 1))
    med = {k: statistics.median(t) for k, t in times.items()}

    bits = lambda x: x.contiguous().view(torch.int32)
    same = {k: bool(torch.equal(bits(state[k + "_fused"][0]), bits(state[k + "_composed"][0])) and
                    torch.equal(state[k + "_fused"][1], state[k + "_composed"][1])) for k in ("hand", "voxel")}
    (gh,) = torch.autograd.grad(hd2, hand_g, g_hand, retain_graph=True)
    td2, tg = state["torch"]
    fd2 = state["hand_fused"][0][:T]
    inside = fd2 > 0
    cmp = {"hands": T, "inside_vertices": int(inside.sum()),
           "depth2_abs_diff_max_m2": float((td2 - fd2).abs().max()),
           "inside_differs": int(((td2 > 0) != inside).sum()),
           "grad_abs_diff_max": float((tg - gh[:T]).abs().max()),
           "grad_abs_max": float(gh[:T].abs().max())}
    a, b = state["refine"]
    res = {"card": name, "power_limit": power, "max_sm_clock": clock,
           "workload": "B=%d closed ellipsoid hands (%d vertices, %d faces) at random poses around an icosphere object of radius "
                       "5 cm (%d faces); pitch %g m -> %d object voxel centres; refinement: synthetic MANO tables (778 vertices, "
                       "%d faces), B=%d" % (B, hv.shape[0], hf.shape[0], of.shape[0], PITCH, C.shape[1], mfaces.shape[0], B),
           "method": "CUDA events around %d calls per stage and 1 torch-arm call, after warm-up; the stages alternate within each of "
                     "%d repetitions; medians" % (args.iters, args.reps),
           "ms": {k: med[k] for k in stages},
           "fused_over_composed": {"hand": med["hand_composed"] / med["hand_fused"],
                                   "voxel": med["voxel_composed"] / med["voxel_fused"]},
           "fused_equals_composed_bitwise": same,
           "inside": {"hand_vertices": int((state["hand_fused"][1] >= 0).sum()),
                      "voxel_centre_hand_pairs": int((state["voxel_fused"][1] >= 0).sum()),
                      "refine_hand_vertices": int((a > 0).sum()), "refine_voxel_pairs": int((b > 0).sum())},
           "torch_fp32_autograd_chunked": {"hands": T, "chunk": args.chunk, "ms": med["torch_autograd"],
                                           "ms_per_hand": med["torch_autograd"] / T,
                                           "dvq_hand_fwd_bwd_ms_per_hand": (med["hand_fused"] + med["hand_backward"]) / B},
           "arms_compared": cmp,
           "ms_all": times}
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()

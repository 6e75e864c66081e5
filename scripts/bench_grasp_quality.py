"""Grasp scoring at the generation batch: B = 4096 closed hand-sized meshes (ellipsoids, 642 vertices / 1280 faces, half-axes
4.5 x 2 x 1.2 cm) at random poses around a ~10 cm object (an icosphere of radius 5 cm, 5120 faces), voxel pitch 5 mm,
contact tolerance 5 mm.  dvq.GraspQuality against a chunked fp32 torch arm on the GPU that does the same arithmetic:

    python scripts/bench_grasp_quality.py [--out profiles/r06_bench_grasp_quality.json] [--reps 5] [--iters 5]

dvq: voxelisation (module construction, once, host clock around a synchronised call), then CUDA events around --iters
calls of each stage after warm-up:
  volume    dvq_mesh_winding of the object's voxel centres against every hand, inside counts only
  inside    dvq_mesh_winding of every hand's vertices against the object
  distance  dvq_mesh_distance of every hand's vertices to the object
  forward   GraspQuality.forward: the three launches plus the device-side reductions (volume, depth, contact)
The torch arm computes the same winding numbers (box rule included), Ericson distances and reductions with broadcast
tensors, chunked over hands; it runs on the first --torch-batch hands (the whole batch would take minutes).  The arms
alternate within each of --reps repetitions; medians are reported, with grasps/s per arm.  The two arms' outputs are
compared on the torch arm's hands.  Prints one JSON line and writes it to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "d-vqvae_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dvq  # noqa: E402
from dvq.grasp_quality import _distance, _winding  # noqa: E402
from test_contact import icosphere  # noqa: E402

B, PITCH, TOL = 4096, 0.005, 0.005


def card():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    return [x.strip() for x in r.stdout.strip().split(",")]


def torch_winding(q, tri, box_lo, box_hi):
    """q [n,Q,3], tri [m,F,3,3] (m = 1 or n) -> w [n,Q] with the box rule"""
    a, b, c = (tri[:, None, :, j, :] - q[:, :, None, :] for j in range(3))
    det = (a * torch.cross(b, c, dim=-1)).sum(-1)
    la, lb, lc = (x.norm(dim=-1) for x in (a, b, c))
    den = la * lb * lc + (a * b).sum(-1) * lc + (b * c).sum(-1) * la + (c * a).sum(-1) * lb
    w = (2 * torch.atan2(det, den)).sum(-1) / (4 * np.pi)
    inb = ((q >= box_lo[:, None]) & (q <= box_hi[:, None])).all(-1)
    return torch.where(inb, w, torch.zeros((), device=q.device))


def torch_distance(q, tri):
    """q [n,Q,3], tri [1,F,3,3] (non-degenerate) -> dist2 [n,Q]: Ericson's cascade as torch.where"""
    a, ab, ac = tri[:, None, :, 0], tri[:, None, :, 1] - tri[:, None, :, 0], tri[:, None, :, 2] - tri[:, None, :, 0]
    ap = q[:, :, None, :] - a
    d1, d2 = (ab * ap).sum(-1), (ac * ap).sum(-1)
    aa, cc, bc = (ab * ab).sum(-1), (ac * ac).sum(-1), (ab * ac).sum(-1)
    d3, d4, d5, d6 = d1 - aa, d2 - bc, d1 - bc, d2 - cc
    vc, vb, va = d1 * d4 - d3 * d2, d5 * d2 - d1 * d6, d3 * d6 - d5 * d4
    z, o = torch.zeros_like(d1), torch.ones_like(d1)
    nv, nw, den = vb, vc, va + vb + vc
    for cond, v_, w_, d_ in reversed([((d1 <= 0) & (d2 <= 0), z, z, o), ((d3 >= 0) & (d4 <= d3), o, z, o),
                                      ((vc <= 0) & (d1 >= 0) & (d3 <= 0), d1, z, d1 - d3), ((d6 >= 0) & (d5 <= d6), z, o, o),
                                      ((vb <= 0) & (d2 >= 0) & (d6 <= 0), z, d2, d2 - d6),
                                      ((va <= 0) & (d4 - d3 >= 0) & (d5 - d6 >= 0), d5 - d6, d4 - d3, (d4 - d3) + (d5 - d6))]):
        nv, nw, den = torch.where(cond, v_, nv), torch.where(cond, w_, nw), torch.where(cond, d_, den)
    r = 1 / den
    d = ap - (nv * r)[..., None] * ab - (nw * r)[..., None] * ac
    return (d * d).sum(-1).nan_to_num(nan=float("inf")).amin(-1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_bench_grasp_quality.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--torch-batch", type=int, default=256)
    ap.add_argument("--chunk", type=int, default=4, help="hands per torch chunk")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_grasp_quality.py measures on the GPU"
    dev = torch.device("cuda:0")
    name, power, clock = card()
    rs = np.random.RandomState(0)
    ov, of = icosphere(0.05, 4)
    hv, hf = icosphere(1.0, 3)
    hv = hv * np.array([0.045, 0.02, 0.012])
    d = rs.randn(B, 3)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rot = np.linalg.qr(rs.randn(B, 3, 3))[0]
    rot *= np.linalg.det(rot)[:, None, None]                             # proper rotations: a reflection would flip w
    hands_np = np.einsum("vk,bjk->bvj", hv, rot) + (rs.uniform(0.0, 0.1, (B, 1)) * d)[:, None, :]
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    obj, hands = cuda(ov), cuda(hands_np)

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gq = dvq.GraspQuality(obj, of, hf, PITCH, TOL).to(dev)
    torch.cuda.synchronize()
    voxel_ms = (time.perf_counter() - t0) * 1e3
    M = gq.num_voxels

    count = torch.zeros(B, device=dev, dtype=torch.int32)
    w = torch.empty(B, hv.shape[0], device=dev)
    state = {}

    def volume():
        count.zero_()
        _winding(gq.centres, hands, gq.hand_faces, count=count)

    def inside():
        _winding(hands, gq.obj_verts, gq.obj_faces, w=w)

    def distance():
        _distance(hands, gq.obj_verts, gq.obj_faces, B)

    def forward():
        state["dvq"] = gq(hands)

    T = args.torch_batch
    obj_tri = obj[torch.from_numpy(of).to(dev)][None]                     # [1, F, 3, 3]
    hf_t = torch.from_numpy(hf).to(dev)
    cen = gq.centres
    olo, ohi = obj.min(0).values[None], obj.max(0).values[None]
    tol2 = torch.tensor(np.float32(np.float32(TOL) * np.float32(TOL)), device=dev)

    def torch_arm():
        out = []
        for b0 in range(0, T, args.chunk):
            h = hands[b0:min(T, b0 + args.chunk)]
            n = h.shape[0]
            cnt = (torch_winding(cen.expand(n, -1, -1), h[:, hf_t], h.min(1).values, h.max(1).values) >= 0.5).sum(1)
            wv = torch_winding(h, obj_tri, olo.expand(n, -1), ohi.expand(n, -1))
            d2 = torch_distance(h, obj_tri)
            ins = wv >= 0.5
            out.append(((cnt.double() * float(np.float32(PITCH)) ** 3).float(),
                        torch.where(ins, d2.sqrt(), torch.zeros((), device=dev)).amax(1), (ins | (d2 <= tol2)).any(1), cnt))
        state["torch"] = [torch.cat(x) for x in zip(*out)]

    stages = {"volume": volume, "inside": inside, "distance": distance, "forward": forward}
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

    times = {k: [] for k in list(stages) + ["torch"]}
    for _ in range(args.reps):
        for k, f in stages.items():
            times[k].append(timed(f, args.iters))
        times["torch"].append(timed(torch_arm, 1))
    med = {k: statistics.median(t) for k, t in times.items()}

    vol, dep, con = (x[:T] for x in state["dvq"])
    tvol, tdep, tcon, tcnt = state["torch"]
    p3 = float(np.float32(PITCH)) ** 3
    cmp = {"hands": T,
           "count_abs_diff_max": int((vol.double() / p3 - tcnt.double()).round().abs().max()),
           "count_differs": int(((vol.double() / p3).round() != tcnt.double()).sum()),
           "depth_abs_diff_max_m": float((dep - tdep).abs().max()),
           "contact_differs": int((con != tcon).sum())}
    full = state["dvq"]
    res = {"card": name, "power_limit": power, "max_sm_clock": clock,
           "workload": "B=%d closed ellipsoid hands (%d vertices, %d faces) at random poses around an icosphere object of radius "
                       "5 cm (%d faces); pitch %g m -> %d object voxel centres (grid %s); contact_tol %g m"
                       % (B, hv.shape[0], hf.shape[0], of.shape[0], PITCH, M, gq.grid, TOL),
           "method": "CUDA events around %d calls per dvq stage and 1 torch-arm call, after warm-up; the arms alternate within each "
                     "of %d repetitions; medians.  Voxelisation: host clock around the synchronised module construction, once"
                     % (args.iters, args.reps),
           "dvq": {"voxelisation_ms_once": voxel_ms,
                   "volume_ms": med["volume"], "inside_ms": med["inside"], "distance_ms": med["distance"],
                   "forward_ms": med["forward"], "grasps_per_s": B / (med["forward"] * 1e-3)},
           "torch_fp32_chunked": {"hands": T, "chunk": args.chunk, "ms": med["torch"], "grasps_per_s": T / (med["torch"] * 1e-3)},
           "speedup_grasps_per_s": (B / med["forward"]) / (T / med["torch"]),
           "outputs": {"penetrating": int((full[1] > 0).sum()), "contact": int(full[2].sum()),
                       "with_volume": int((full[0] > 0).sum()), "mean_volume_cm3": float(full[0].double().mean() * 1e6)},
           "arms_compared": cmp,
           "ms_all": times}
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()

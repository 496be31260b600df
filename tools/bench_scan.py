"""Timing of sceneego_voxelize_scan: one world-space scan seen from B camera poses -> B occupancy grids in one launch.

    python tools/bench_scan.py [--batch 64] [--volume 64] [--points 4194304,16777216] [--sides 2.0,2.5]
                               [--repeats 7] [--out profiles/...json]

Workload: a synthetic room scan (utils/synth.synthetic_world_scan: floor, walls, ceiling and four boxes; N points) and
a head-mounted camera's trajectory of B poses through the room (synthetic_head_trajectory), fp64 and fp32.  16 M points
(384 MB in fp64) exceed the 126 MB L2; for every size the L2 is overwritten before each timed window anyway, so the
scan comes from HBM.  CUDA events around the C entry point alone (no host-side argument checks in the window); median
of the repeats.  The grids' zeroing, which the caller owes either route, is outside both windows.

Compared in the same process, alternating with the fused kernel repeat by repeat:
  (a) what a user writes without it: each frame's cloud transformed in torch (A[k,0]*x + A[k,1]*y + A[k,2]*z + t[k],
      elementwise, the same operation order), `--chunk` frames at a time, then one sceneego_voxelize_points launch per
      chunk.  Its grids must equal the fused kernel's, bit for bit (asserted).
  (b) the NumPy restatement (tests/scan_oracle.voxelize_scan) on one frame: the host route.
Ablation, also event-timed: the same launch with every pose moved 1 km away, so no point lands in any cuboid: the
transform, the quantisation and the writer election still run, the stores do not.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from sceneego_b200 import _lib  # noqa: E402
from sceneego_b200.utils import synth  # noqa: E402
from tests import scan_oracle as sco  # noqa: E402

FRAME_TILE = 32          # kScanFrameTile in csrc/geometry.cu: the scan is read once per tile of frames


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip() or r.stderr.strip()}


def ev_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def med(xs):
    return sorted(xs)[len(xs) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--volume", type=int, default=64)
    ap.add_argument("--points", default="4194304,16777216")
    ap.add_argument("--sides", default="2.0,2.5")
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--chunk", type=int, default=8, help="frames per transformed-cloud chunk of route (a)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_scan needs a CUDA device")
    B, V = a.batch, a.volume
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")     # 4x the L2
    res = {"gpu": gpu_info(), "batch": B, "volume_size": V, "repeats": a.repeats, "route_a_chunk_frames": a.chunk,
           "frame_tile": FRAME_TILE,
           "timing": "CUDA events around one call, L2 overwritten before each window, median; fused and route (a) "
                     "alternate repeat by repeat", "runs": []}
    poses64 = synth.synthetic_head_trajectory(B, seed=2)
    far = poses64.copy()
    far[:, 2, 3] -= 1000.0                                                # every cuboid 1 km behind its camera
    for n in [int(x) for x in a.points.split(",")]:
        scan64_np = synth.synthetic_world_scan(n, seed=1)
        for dt_name, dt_np, dt in (("float64", np.float64, torch.float64), ("float32", np.float32, torch.float32)):
            scan_np = scan64_np.astype(dt_np)
            scan = torch.from_numpy(scan_np).cuda()
            x, y, z = scan[:, 0], scan[:, 1], scan[:, 2]
            pose_np = poses64.astype(dt_np)
            pose = torch.from_numpy(pose_np).cuda()
            d_pose = pose[:, :3, :].contiguous()
            d_far = torch.from_numpy(far.astype(dt_np)[:, :3, :].copy()).cuda()
            is64 = int(dt == torch.float64)
            for s in [float(v) for v in a.sides.split(",")]:
                occ = torch.zeros(B, V, V, V, dtype=torch.float32, device="cuda")
                occ_a = torch.zeros_like(occ)
                k = a.chunk
                offs = torch.arange(k + 1, dtype=torch.int64, device="cuda") * n
                cams = torch.empty(k * n, 3, dtype=dt, device="cuda")

                def fused(p=d_pose):
                    _lib._call("sceneego_voxelize_scan", scan, scan, is64, C.c_int64(n), p, B, V, C.c_double(s), occ)

                def route_a():
                    for b0 in range(0, B, k):
                        m = min(k, B - b0)
                        cv = cams[:m * n].view(m, n, 3)
                        for j in range(m):
                            P = pose[b0 + j]
                            for c in range(3):
                                torch.add(P[c, 0] * x + P[c, 1] * y + P[c, 2] * z, P[c, 3], out=cv[j, :, c])
                        _lib._call("sceneego_voxelize_points", cams, cams, is64, offs[:m + 1], m, V, C.c_double(s),
                                   occ_a[b0:b0 + m])

                fused()
                route_a()                                                  # warm-up (module load, allocator)
                torch.cuda.synchronize()
                assert torch.equal(occ, occ_a), (n, dt_name, s)
                t_fused, t_a, t_far = [], [], []
                for _ in range(a.repeats):
                    flush.zero_()
                    t_fused.append(ev_ms(fused))
                    flush.zero_()
                    t_a.append(ev_ms(route_a))
                    flush.zero_()
                    t_far.append(ev_ms(lambda: fused(d_far)))
                occ.zero_()
                fused()
                occ_a.zero_()
                route_a()
                torch.cuda.synchronize()
                exact_a = bool(torch.equal(occ, occ_a))
                assert exact_a, (n, dt_name, s)
                # point-frames inside the cuboid (|x|, |y| <= s/2, 0 <= z <= s in the camera frame)
                inside = 0
                h = s / 2
                for P in pose:
                    c0 = P[0, 0] * x + P[0, 1] * y + P[0, 2] * z + P[0, 3]
                    c1 = P[1, 0] * x + P[1, 1] * y + P[1, 2] * z + P[1, 3]
                    c2 = P[2, 0] * x + P[2, 1] * y + P[2, 2] * z + P[2, 3]
                    inside += int(((c0.abs() <= h) & (c1.abs() <= h) & (c2 >= 0) & (c2 <= s)).sum().item())
                # (b) the host restatement, one frame, and its agreement with the kernel
                i = B // 3
                t0 = time.perf_counter()
                want = sco.voxelize_scan(scan_np, pose_np[i:i + 1], V, s)[0]
                host_ms = (time.perf_counter() - t0) * 1000.0
                exact_np = bool(np.array_equal(occ[i].cpu().numpy(), want))
                assert exact_np, (n, dt_name, s)
                mf, ma, mfar = med(t_fused), med(t_a), med(t_far)
                scan_bytes = n * 3 * scan.element_size()
                tiles = (B + FRAME_TILE - 1) // FRAME_TILE
                run = {"points": n, "dtype": dt_name, "cuboid_side": s,
                       "fused_ms": mf, "fused_ms_all": t_fused, "us_per_frame": 1000.0 * mf / B,
                       "Gpoint_frames_per_s": n * B / mf / 1e6,
                       "scan_bytes": scan_bytes, "scan_reads": tiles,
                       "scan_GB_read_per_s": scan_bytes * tiles / mf / 1e6,
                       "fraction_point_frames_in_cuboid": inside / (n * B),
                       "occupied_voxels_per_frame": float(occ.sum().item()) / B,
                       "no_hit_ablation_ms": mfar, "no_hit_ablation_ms_all": t_far,
                       "route_a_torch_transform_then_voxelize_points_ms": ma, "route_a_ms_all": t_a,
                       "route_a_us_per_frame": 1000.0 * ma / B, "speedup_vs_route_a": ma / mf,
                       "route_a_bit_exact": exact_a,
                       "host_numpy_ms_per_frame": host_ms, "speedup_vs_host_numpy_per_frame": host_ms / (mf / B),
                       f"frame{i}_bit_exact_vs_numpy": exact_np}
                res["runs"].append(run)
                print(json.dumps({k_: v for k_, v in run.items() if not k_.endswith("_all")}), flush=True)
                del occ, occ_a, cams
            del scan, x, y, z
        torch.cuda.empty_cache()
    res["host_cpu_threads"] = torch.get_num_threads()
    line = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    print(json.dumps({"gpu": res["gpu"], "runs": len(res["runs"])}))


if __name__ == "__main__":
    main()

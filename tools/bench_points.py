"""Timing of the point-cloud scatter sceneego_voxelize_points (point_cloud_to_voxel_numpy,
network/voxel_net_depth.py:207-222) on one GPU.

    python tools/bench_points.py [--batch 64] [--volume 64] [--repeats 7] [--out profiles/...json]

Workload: B synthetic room clouds (utils/synth.synthetic_depth_room x the fp64 ray table, row-major, 1,310,720 points
per frame including the zero-depth ones outside the image circle, which all land on one voxel), as float64 and as
float32 clouds.  CUDA events around the kernel alone (the C entry point, no host-side argument checks in the window);
the 126 MB L2 is overwritten between repeats so the points come from HBM; median of the repeats.  The zeroing of the
occupancy grid the caller owes the kernel is timed on its own.  Baseline: the host NumPy restatement of the reference
(tests/points_oracle.voxelize_points), per frame, on the same clouds -- what a user of the reference pays per frame today.
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
from sceneego_b200.utils.fisheye.FishEyeCalibrated import FishEyeCameraCalibrated  # noqa: E402
from tests import points_oracle as pto  # noqa: E402

DATASHEET_HBM_GBS = 7700.0     # HGX B200 data sheet, one GPU


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip() or r.stderr.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--volume", type=int, default=64)
    ap.add_argument("--side", type=float, default=2.0)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--cpu-frames", type=int, default=2, help="frames timed through the host NumPy oracle")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_points needs a CUDA device")
    B, V, s = a.batch, a.volume, a.side
    cam = FishEyeCameraCalibrated(os.path.join(ROOT, "sceneego_b200", "data", "fisheye.calibration_05_08.json"))
    ray_dev = cam.ray_table_device(1280, 1024, "cuda")
    ray_np = ray_dev.permute(1, 0, 2).reshape(-1, 3).cpu().numpy()
    depth = synth.synthetic_depth_room(B, ray_np, seed=7).cuda()
    n_frame = 1024 * 1280
    pts64 = (ray_dev.unsqueeze(0) * depth.double().unsqueeze(-1)).reshape(-1, 3).contiguous()
    pts32 = pts64.float()
    offsets = torch.arange(B + 1, dtype=torch.int64, device="cuda") * n_frame
    occ = torch.zeros(B, V, V, V, dtype=torch.float32, device="cuda")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")     # 4x the L2
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peaks = json.load(open(peaks_path)) if os.path.exists(peaks_path) else {}
    hbm = float(peaks.get("hbm_gbs", DATASHEET_HBM_GBS))
    res = {"gpu": gpu_info(), "batch": B, "points_per_frame": n_frame, "volume_size": V, "cuboid_side": s,
           "repeats": a.repeats, "timing": "CUDA events around one launch, L2 overwritten before each repeat, median",
           "hbm_GB_per_s_reference": hbm,
           "hbm_reference_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "HGX B200 data sheet"}

    def ev_ms(fn):
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a_.record()
        fn()
        b_.record()
        torch.cuda.synchronize()
        return a_.elapsed_time(b_)

    memset_ms = []
    for name, pts in (("float64", pts64), ("float32", pts32)):
        launch = lambda: _lib._call("sceneego_voxelize_points", pts, pts, int(pts.dtype == torch.float64), offsets, B, V,
                                    C.c_double(s), occ)
        occ.zero_()
        launch()                                                           # warm-up (module load)
        torch.cuda.synchronize()
        ms = []
        for _ in range(a.repeats):
            memset_ms.append(ev_ms(occ.zero_))
            flush.zero_()
            torch.cuda.synchronize()
            ms.append(ev_ms(launch))
        med = sorted(ms)[len(ms) // 2]
        occupied = int(occ.sum().item())
        # algorithmic bytes: every point read once, one 4-byte store per occupied voxel
        read_b = pts.numel() * pts.element_size()
        write_b = 4 * occupied
        # the kernel against the NumPy restatement of the reference on one frame
        i = B // 2
        want = pto.voxelize_points(pts[i * n_frame:(i + 1) * n_frame].cpu().numpy(), V, s)
        exact = bool(np.array_equal(occ[i].cpu().numpy(), want))
        res[name] = {"kernel_ms": med, "kernel_ms_all": ms, "us_per_frame": 1000.0 * med / B,
                     "Gpoints_per_s": B * n_frame / med / 1e6,
                     "algorithmic_bytes": {"points_read": read_b, "occupancy_written": write_b,
                                           "grid_memset_separate": B * V ** 3 * 4},
                     "GB_per_s": (read_b + write_b) / med / 1e6,
                     "fraction_of_hbm_reference": (read_b + write_b) / med / 1e6 / hbm,
                     "hbm_bound_us_per_frame": (read_b + write_b) / B / (hbm * 1e9) * 1e6,
                     "occupied_voxels_per_frame": occupied / B,
                     f"frame{i}_bit_exact_vs_numpy_oracle": exact}
        # host baseline: the reference's NumPy on the same clouds, per frame
        host = [pts[j * n_frame:(j + 1) * n_frame].cpu().numpy() for j in range(a.cpu_frames)]
        pto.voxelize_points(host[0], V, s)
        t0 = time.perf_counter()
        for h in host:
            pto.voxelize_points(h, V, s)
        res[name]["host_numpy_ms_per_frame"] = (time.perf_counter() - t0) * 1000.0 / len(host)
        res[name]["speedup_vs_host_numpy_per_frame"] = res[name]["host_numpy_ms_per_frame"] / (med / B)
    res["grid_memset_ms_median"] = sorted(memset_ms)[len(memset_ms) // 2]
    res["host_cpu_threads"] = torch.get_num_threads()
    line = json.dumps(res, indent=1)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

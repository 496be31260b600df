"""Cost of a camera per frame: the camera-per-frame gather and depth voxelisation against the single-camera kernels, and
whole-`lift()` throughput with and without `camera_ids`.

    python tools/bench_cameras.py [--batch 64] [--volume 64] [--repeats 15] [--lift-steps 10] [--out profiles/...json]

Workload: B frames of (64,64,32) features and 1024x1280 room depth maps, V^3 voxels, the z-window input layout of the
marching stem (the bench configuration: the gather writes the 16-bit volume, the voxelisation the plain f32 grid that
occ_expand_zwin turns into the occupancy plane).  Cameras: the 05_08 calibration and K - 1 variants of it (image centre
shifted by a few pixels, polynomial coefficients scaled by a few per cent), K in {1, 2, 4, 8}; camera assignments: all
equal, sorted, interleaved (b mod K) and random, each visited in the stable frame order lift() passes.

Kernel times: CUDA events around one call, the L2 overwritten before every window (inside lift() the V2V program runs
between two batches' gathers, so their inputs do not stay in L2), median of the repeats; the single-camera kernels and
the camera-per-frame kernels alternate repeat by repeat.  Every camera-per-frame result is compared with one
single-camera launch per camera first.  lift(): `--lift-steps` calls after a warm-up, with a device synchronise at
both ends of the window, output #2 off; the camera-per-frame runs use K = 4 with random ids.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from sceneego_b200 import DEFAULT_CALIBRATION, _lib  # noqa: E402
from sceneego_b200.network.voxel_net_depth import VoxelNetwork_depth, camera_frame_order  # noqa: E402
from sceneego_b200.utils import cfg as cfgmod, synth  # noqa: E402
from sceneego_b200.utils.fisheye.FishEyeCalibrated import FishEyeCameraCalibrated  # noqa: E402

IMG_H, IMG_W = 1024, 1280


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


def calib_files(tmp, k_max):
    base = json.load(open(DEFAULT_CALIBRATION))
    files = [DEFAULT_CALIBRATION]
    for k in range(1, k_max):
        d = json.loads(json.dumps(base))
        d["intrinsic"][0][2] += 1.5 * k - 6.0
        d["intrinsic"][1][2] += 4.0 - 1.25 * k
        d["polynomialC2W"] = [c * (1.0 + 0.006 * k) for c in d["polynomialC2W"]]
        d["polynomialW2C"] = [c * (1.0 - 0.004 * k) for c in d["polynomialW2C"]]
        p = os.path.join(tmp, f"cam{k}.json")
        json.dump(d, open(p, "w"))
        files.append(p)
    return files


def assignment(kind, B, K, rng):
    if kind == "equal":
        return np.zeros(B, np.int32)
    if kind == "sorted":
        return np.sort(np.arange(B) % K).astype(np.int32)
    if kind == "interleaved":
        return (np.arange(B) % K).astype(np.int32)
    return rng.integers(0, K, B).astype(np.int32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--volume", type=int, default=64)
    ap.add_argument("--cameras", default="1,2,4,8")
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--lift-steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cameras needs a CUDA device")
    B, V = a.batch, a.volume
    ks = [int(k) for k in a.cameras.split(",")]
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")      # 4x the L2
    rng = np.random.default_rng(0)
    tmp = tempfile.mkdtemp(prefix="bench_cameras_")
    files = calib_files(tmp, max(max(ks), 4))
    models = [FishEyeCameraCalibrated(f) for f in files]
    calibs = [m.calib_struct(IMG_W, IMG_H) for m in models]
    grids_all = torch.stack([_lib.project_voxels(c, V, 2.0, (IMG_H, IMG_W), "cuda")[1] for c in calibs])
    rays_all = torch.stack([_lib.ray_table(c, "cuda") for c in calibs])
    g = torch.Generator().manual_seed(1)
    feat = torch.randn(B, 64, 64, 32, generator=g).cuda()
    ray0 = rays_all[0].permute(1, 0, 2).reshape(-1, 3).cpu().numpy()
    depth = synth.synthetic_depth_room(B, ray0, seed=3).cuda()
    lay = _lib.vol_layout_zwin(V, B)
    vol = _lib.alloc_volume(lay, 40, "cuda")
    vol_ref = _lib.alloc_volume(lay, 40, "cuda")
    occ = torch.zeros(B, V, V, V, device="cuda")
    occ_ref = torch.zeros_like(occ)
    res = {"gpu": gpu_info(), "batch": B, "volume_size": V, "layout": "z-window (marching stem input)",
           "repeats": a.repeats,
           "timing": "CUDA events around one call, L2 overwritten before each window, median; single-camera and "
                     "camera-per-frame kernels alternate repeat by repeat; us_per_frame = median / batch",
           "cameras": "05_08 and K-1 variants: centre shifted by a few px, polynomials scaled by a few per cent",
           "kernels": []}

    def single(kind):
        if kind == "voxelize":
            return lambda: _lib.voxelize_depth(depth, rays_all[0], IMG_H, IMG_W, V, 2.0, occ_ref, None, None)
        fused = kind == "gather_fused"
        return lambda: _lib.unproject(feat, None if fused else grids_all[0], calibs[0] if fused else None, V, 2.0,
                                      IMG_H, IMG_W, None, vol_ref, lay, extra_zero_planes=1)

    def per_frame(kind, K, d_ids, d_order):
        if kind == "voxelize":
            rays = rays_all[:K].contiguous()
            return lambda: _lib.voxelize_depth_cameras(depth, None, float("inf"), rays, d_ids, d_order, IMG_H, IMG_W, V,
                                                       2.0, occ, None, None)
        fused = kind == "gather_fused"
        grids = grids_all[:K].contiguous()
        return lambda: _lib.unproject_cameras(feat, None if fused else grids, calibs[:K], d_ids, d_order, V, 2.0, IMG_H,
                                              IMG_W, None, vol, lay, extra_zero_planes=1)

    def check(kind, K, ids, fn):
        """the camera-per-frame result equals one single-camera launch per camera (all frames, camera by camera)"""
        occ.zero_()
        fn()
        for k in range(K):
            fk = torch.from_numpy(np.nonzero(ids == k)[0]).cuda()
            if fk.numel() == 0:
                continue
            if kind == "voxelize":
                o = torch.zeros(fk.numel(), V, V, V, device="cuda")
                _lib.voxelize_depth(depth[fk].contiguous(), rays_all[k].contiguous(), IMG_H, IMG_W, V, 2.0, o, None, None)
                assert torch.equal(occ[fk], o), (kind, K, k)
            else:
                fused = kind == "gather_fused"
                o = torch.empty(fk.numel(), 32, V, V, V, device="cuda")
                _lib.unproject(feat[fk].contiguous(), None if fused else grids_all[k].contiguous(),
                               calibs[k] if fused else None, V, 2.0, IMG_H, IMG_W, o, None, None)
                got = _lib.unpack_volume(vol, lay, B, 32)[fk]
                assert torch.equal(got, o.to(_lib.act_torch_dtype()).float()), (kind, K, k)
        occ.zero_()

    for kind in ("gather_table", "gather_fused", "voxelize"):
        base = single(kind)
        base()
        for K in ks:
            for pat in (["equal"] if K == 1 else ["equal", "sorted", "interleaved", "random"]):
                ids = assignment(pat, B, K, rng)
                d_ids = torch.from_numpy(ids).cuda()
                d_order = torch.from_numpy(camera_frame_order(ids)).cuda()
                fn = per_frame(kind, K, d_ids, d_order)
                check(kind, K, ids, fn)
                t_single, t_cam = [], []
                for _ in range(a.repeats):
                    flush.zero_()
                    t_single.append(ev_ms(base))
                    flush.zero_()
                    t_cam.append(ev_ms(fn))
                run = {"kernel": kind, "cameras": K, "ids": pat, "camera_changes_in_order": int(len(set(ids)) - 1),
                       "single_camera_us_per_frame": med(t_single) * 1000.0 / B,
                       "camera_per_frame_us_per_frame": med(t_cam) * 1000.0 / B}
                run["ratio"] = run["camera_per_frame_us_per_frame"] / run["single_camera_us_per_frame"]
                print(json.dumps(run), flush=True)
                res["kernels"].append(run)

    # whole lift(): the bench configuration (one 64-frame V2V chunk), output #2 off
    with contextlib.redirect_stdout(io.StringIO()):
        net = VoxelNetwork_depth(cfgmod.default_config(batch_size=B, volume_size=V), device="cuda", v2v_chunk=B,
                                 materialize_features=False).eval()
        for f in files[1:4]:
            net.add_camera(f)
    sd = synth.synthetic_state_dict(synth.stage_state_shapes(), seed=0, mode="random_bn")
    full = net.state_dict()
    full.update(sd)
    net.load_state_dict(full, strict=True)
    feat256 = synth.synthetic_features(B, seed=5).cuda()
    lift_runs = []
    cases = [("none", None), ("random K=4", assignment("random", B, 4, rng)), ("sorted K=4", assignment("sorted", B, 4, rng))]
    with torch.no_grad():
        for name, ids in cases:                                          # warm-up every configuration
            net.lift(feat256, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=depth, camera_ids=ids)
        for rep in range(3):                                             # alternate the configurations
            for name, ids in cases:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(a.lift_steps):
                    net.lift(feat256, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=depth,
                             camera_ids=ids)
                torch.cuda.synchronize()
                lift_runs.append({"camera_ids": name, "round": rep,
                                  "frames_per_s": B * a.lift_steps / (time.perf_counter() - t0)})
                print(json.dumps(lift_runs[-1]), flush=True)
    res["lift"] = {"config": f"batch {B}, v2v_chunk {B}, V {V}, output #2 off, table-mode gather, depth_map_batch",
                   "steps_per_round": a.lift_steps, "runs": lift_runs,
                   "median_frames_per_s": {n: med([r["frames_per_s"] for r in lift_runs if r["camera_ids"] == n])
                                           for n, _ in cases}}
    res["gpu_after"] = gpu_info()
    print(json.dumps(res["lift"]["median_frames_per_s"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

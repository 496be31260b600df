"""Dataset-side depth handling on the GPU (reference: dataset/real_depth_utils.py:29-60,
dataset/demo_dataset.py:86-96, dataset/test_dataset.py:138-148).

The reference's datasets decode an EXR, nearest-resize it to 1280x1024 when needed, clamp depth > 10 m to 10 m and
-- with `voxel_output=True` -- turn it into a (V,V,V) occupancy grid on the host with `depth_map_to_voxel`.  Here the
resize, the clamp and the voxelisation are ONE kernel launch over a batch of raw maps
(`sceneego_voxelize_depth_dataset_f64`); EXR decoding stays host I/O.  Same function names and argument meaning as
the reference; tensors live on the CUDA device.

NOTE the dataset's `depth_map_to_voxel` is NOT the network's `depth_map_to_voxel_numpy`
(network/voxel_net_depth.py:194-205): it multiplies the full 1280-wide map by the ray table pixel for pixel, without
the network's nearest squash to 1024x1024 and its 128 zero-padded columns (7,782 vs 8,331 occupied voxels on the
demo frame img_001000).  Both are provided, each pinned against the reference function it replaces
(tests/golden/voxel_dataset.npz, tests/golden/voxel.npz).

Clouds that do not come from a depth map (a reconstructed mesh, SLAM, a LiDAR sweep) enter through
`point_cloud_to_voxel_pytorch` (one cloud, :45-60) or `point_clouds_to_voxels` (a ragged batch, one launch of
`sceneego_voxelize_points`); the grids go to the network as `scene_volumes=`.  A static world-space scan with one
camera pose per frame enters through `scan_to_voxels` (one launch of `sceneego_voxelize_scan`, no per-frame copy of
the scan).
"""
from __future__ import annotations

import weakref

import numpy as np
import torch

from .. import _lib

PRE_H, PRE_W, CLAMP_MAX = 1024, 1280, 10.0     # demo_dataset.py:87-91

_RAY_CACHE_MAX = 4
_ray_cache = []      # [(weakref to the source array | None, source array id, device str, device tensor)]


def _device_ray(ray, device, image_width=PRE_W, image_height=PRE_H) -> torch.Tensor:
    """The reference's ray table is a NumPy (W*H, 3) array in x-major order (network/voxel_net_depth.py:147-155);
    the kernel reads a row-major (H, W, 3) fp64 device table.  Converted once per live source array: the cache
    entry holds a weak reference to the array, so a different table that happens to reuse its id() after garbage
    collection is never mistaken for it, and at most _RAY_CACHE_MAX tables are kept."""
    if isinstance(ray, torch.Tensor) and ray.is_cuda and ray.dim() == 3:
        return ray
    dev = str(_lib._as_device(device))
    for ref, rid, d, t in _ray_cache:
        if d == dev and rid == id(ray) and ref is not None and ref() is ray:
            return t
    arr = np.asarray(ray.detach().cpu() if isinstance(ray, torch.Tensor) else ray, dtype=np.float64)
    arr = arr.reshape(image_width, image_height, 3)
    t = torch.from_numpy(np.ascontiguousarray(arr.transpose(1, 0, 2))).to(dev)
    try:
        ref = weakref.ref(ray)
    except TypeError:
        ref = None                               # not weak-referenceable (e.g. a list): converted on every call
    if ref is not None:
        _ray_cache[:] = [e for e in _ray_cache if e[0] is not None and e[0]() is not None][-(_RAY_CACHE_MAX - 1):]
        _ray_cache.append((ref, id(ray), dev, t))
    return t


def depth_maps_to_voxels(ray, depth_raw: torch.Tensor, cuboid_side: float, volume_size: int,
                         preprocess: bool = True, network_semantics: bool = False) -> torch.Tensor:
    """Batch form of `depth_map_to_voxel`: depth_raw (B,h,w) f32 CUDA -> (B,V,V,V) f32 {0,1}.
    preprocess=True fuses the dataset's resize to 1280x1024 and the 10 m clamp (demo_dataset.py:86-91) into the load;
    False expects maps that are already 1024x1280 and clamped.
    network_semantics=True gives what the NETWORK computes from the same map (voxel_net_depth.py:194-222: squash to
    1024x1024, 128 padded columns) -- the grids to pass as `scene_volumes=` for results identical to
    `depth_map_batch=`."""
    if not depth_raw.is_cuda:
        raise _lib.SceneEgoError("depth_maps_to_voxels needs CUDA tensors (no CPU fallback)")
    d = depth_raw.contiguous().float()
    b = d.shape[0]
    occ = torch.zeros(b, volume_size, volume_size, volume_size, dtype=torch.float32, device=d.device)
    r = _device_ray(ray, d.device)
    if not preprocess and tuple(d.shape[1:]) != (PRE_H, PRE_W):
        raise _lib.SceneEgoError(f"preprocess=False expects ({PRE_H}, {PRE_W}) maps (the ray table's size), got "
                                 f"{tuple(d.shape[1:])}")
    clamp = CLAMP_MAX if preprocess else float("inf")
    if network_semantics:
        _lib.voxelize_depth_raw(d, (PRE_H, PRE_W), clamp, r, PRE_H, PRE_W, volume_size, float(cuboid_side), occ,
                                None, None)
    else:
        _lib.voxelize_depth_dataset(d, (PRE_H, PRE_W), clamp, r, volume_size, float(cuboid_side), occ)
    return occ


def point_clouds_to_voxels(points, counts_or_offsets, cuboid_side: float, volume_size: int) -> torch.Tensor:
    """Batch form of `point_cloud_to_voxel_pytorch` (one launch of `sceneego_voxelize_points`): a ragged batch of
    camera-space clouds -> (B,V,V,V) f32 {0,1} on the clouds' device.

    points: one (N,3) float64 / float32 CUDA tensor holding every frame's points back to back, or a list of (N_b,3)
        tensors (concatenated on the device; they must share a dtype).  The arithmetic follows the dtype, like NumPy
        and torch: float32 clouds are quantised in fp32, float64 clouds in fp64.
    counts_or_offsets: B per-frame point counts, or B+1 offsets (frame b owns points [offsets[b], offsets[b+1])), as a
        sequence, array or tensor.  Entries that sum to N are read as counts; otherwise they must be offsets (0 first,
        N last, non-decreasing).  The two readings only collide for [0, ..., 0, N], which is read as counts.  None with
        a list of clouds takes the list's lengths."""
    if isinstance(points, (list, tuple)):
        clouds = [torch.as_tensor(p) for p in points]
        if not clouds:
            raise _lib.SceneEgoError("point_clouds_to_voxels: empty list of clouds (pass a (0,3) tensor and counts)")
        if any(c.dtype != clouds[0].dtype for c in clouds):
            raise _lib.SceneEgoError("point_clouds_to_voxels: the clouds of a batch must share a dtype")
        if counts_or_offsets is None:
            counts_or_offsets = [c.reshape(-1, 3).shape[0] for c in clouds]
        points = torch.cat([c.reshape(-1, 3) for c in clouds]) if len(clouds) > 1 else clouds[0]
    if not isinstance(points, torch.Tensor) or not points.is_cuda:
        raise _lib.SceneEgoError("point_clouds_to_voxels needs CUDA tensors (no CPU fallback)")
    if counts_or_offsets is None:
        raise _lib.SceneEgoError("point_clouds_to_voxels: per-frame counts or offsets are required with one tensor")
    c = torch.as_tensor(counts_or_offsets).reshape(-1).to("cpu", torch.int64)
    n = points.shape[0] if points.dim() == 2 else -1
    if int(c.sum()) == n and not bool((c < 0).any()):
        offsets = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(c, 0)])
    elif c.numel() >= 1 and int(c[0]) == 0 and int(c[-1]) == n and bool((c[1:] >= c[:-1]).all()):
        offsets = c
    else:
        raise _lib.SceneEgoError(f"point_clouds_to_voxels: need B counts >= 0 summing to {n} points, or B+1 "
                                 f"non-decreasing offsets from 0 to {n}")
    v = int(volume_size)
    occ = torch.zeros(offsets.numel() - 1, v, v, v, dtype=torch.float32, device=points.device)
    _lib.voxelize_points(points.contiguous(), offsets, v, float(cuboid_side), occ)
    return occ


def scan_to_voxels(scan, cam_from_world, cuboid_side: float, volume_size: int) -> torch.Tensor:
    """One static world-space scan (a mesh, SLAM map or LiDAR sweep of the room) seen from B camera poses -> (B,V,V,V)
    f32 {0,1}, one launch of `sceneego_voxelize_scan`; the per-frame transformed clouds are never materialised.

    scan: (N,3) float64 / float32 CUDA tensor; the transform and the quantisation run in its precision.
    cam_from_world: (B,4,4) poses of the scan's dtype (CPU or CUDA) mapping world points into the camera frame that
        ray x depth produces; frame b's grid is `point_cloud_to_voxel_pytorch` of
        `A[k,0]*x + A[k,1]*y + A[k,2]*z + t[k]` (that order, no FMA) with [A|t] = cam_from_world[b, :3]."""
    if not isinstance(scan, torch.Tensor) or not scan.is_cuda:
        raise _lib.SceneEgoError("scan_to_voxels needs a CUDA scan tensor (no CPU fallback)")
    pose = torch.as_tensor(cam_from_world)
    v = int(volume_size)
    occ = torch.zeros(pose.shape[0] if pose.dim() == 3 else 0, v, v, v, dtype=torch.float32, device=scan.device)
    _lib.voxelize_scan(scan.contiguous(), pose, v, float(cuboid_side), occ)
    return occ


def point_cloud_to_voxel_pytorch(scene_point_cloud, cuboid_side, volume_size):
    """dataset/real_depth_utils.py:45-60 for ONE camera-space cloud: (N,3) float64 / float32 tensor or array (CPU
    inputs are copied to the current CUDA device) -> (V,V,V) f32 {0,1}.  Argument order (cloud, cuboid side, volume
    size) as `depth_map_to_voxel` calls it (:29-43).  The quantisation runs in the cloud's precision."""
    p = torch.as_tensor(scene_point_cloud)
    if not p.is_cuda:
        p = p.cuda()
    p = p.reshape(-1, 3)
    return point_clouds_to_voxels(p, [p.shape[0]], cuboid_side, volume_size)[0]


def depth_map_to_voxel(ray, depth, cuboid_side, volume_size):
    """dataset/real_depth_utils.py:29-43, one PREPROCESSED (1024,1280) map (what the reference's datasets pass):
    point cloud = ray table x depth, pixel for pixel; quantised and scattered like :45-60."""
    d = torch.as_tensor(depth)
    if not d.is_cuda:
        d = d.cuda()
    return depth_maps_to_voxels(ray, d.reshape(1, d.shape[-2], d.shape[-1]), cuboid_side, volume_size,
                                preprocess=False)[0]

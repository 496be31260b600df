"""CPU restatement of point_cloud_to_voxel_numpy (network/voxel_net_depth.py:207-222; twin of
dataset/real_depth_utils.py:45-60) for the point-cloud tests and tools/bench_points.py.  Checker side only: pinned to
the reference-generated depth goldens through oracle.sceneego_oracle.voxelize_depth / voxelize_depth_dataset
(tests/test_points_voxel.py)."""
import numpy as np


def voxelize_points(points: np.ndarray, volume_size: int, cuboid_side: float) -> np.ndarray:
    """One camera-space (N,3) cloud -> (V,V,V) f32 {0,1}.

    The caller's dtype is kept, as the reference keeps it: a float64 cloud is computed in fp64, a float32 cloud in fp32
    (float32 array + Python float stays float32 under NumPy 1.x value-based casting and NumPy 2 / NEP 50 alike).
    q_xy = ((p + s/2) * V) / s, q_z = (p_z * V) / s, round half-to-even, keep iff 0 <= q <= V-1 on all axes.
    """
    V, s = int(volume_size), float(cuboid_side)              # Python scalars: they never widen the cloud's dtype
    pc = np.array(points, copy=True).reshape(-1, 3)          # copy(scene_point_cloud): the caller's dtype
    with np.errstate(invalid="ignore", over="ignore"):       # inf / NaN / overflowing points are dropped below
        pc[:, 0] = (pc[:, 0] + s / 2) * V / s
        pc[:, 1] = (pc[:, 1] + s / 2) * V / s
        pc[:, 2] = pc[:, 2] * V / s
        q = np.round(pc)
        ok = np.all(np.logical_and(V - 1 >= q, q >= 0), axis=1)
    qi = q[ok].astype(np.int64)
    vox = np.zeros((V, V, V), dtype=np.float32)
    vox[qi[:, 0], qi[:, 1], qi[:, 2]] = 1.0
    return vox

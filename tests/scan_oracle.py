"""CPU restatement of sceneego_voxelize_scan (one world-space scan seen from per-frame camera poses) on top of
tests/points_oracle.voxelize_points, for tests/test_scan_voxel.py and tools/bench_scan.py.  Checker side only: pinned
to voxelize_points and, through signed-permutation poses, to the reference-generated depth goldens
(tests/test_scan_voxel.py)."""
import numpy as np

from tests.points_oracle import voxelize_points


def voxelize_scan(scan: np.ndarray, cam_from_world: np.ndarray, volume_size: int, cuboid_side: float) -> np.ndarray:
    """One world-space (N,3) scan seen from B (4,4) cam_from_world poses -> (B,V,V,V) f32 {0,1}: frame b is
    voxelize_points of c_k = A[k,0]*x + A[k,1]*y + A[k,2]*z + t[k] with [A|t] = cam_from_world[b, :3].

    Elementwise NumPy operations in the scan's dtype, evaluated left to right with every product and sum rounded
    (no `@` / einsum / dot: BLAS may contract to FMA).  The poses must have the scan's dtype."""
    scan = np.asarray(scan).reshape(-1, 3)
    pose = np.asarray(cam_from_world)
    assert pose.dtype == scan.dtype and pose.ndim == 3 and pose.shape[1:] == (4, 4)
    x, y, z = scan[:, 0], scan[:, 1], scan[:, 2]
    out = np.zeros((pose.shape[0],) + (int(volume_size),) * 3, dtype=np.float32)
    for b, P in enumerate(pose):
        c = np.empty_like(scan)
        with np.errstate(invalid="ignore", over="ignore"):    # inf * 0 -> NaN and overflow: dropped as in voxelize_points
            for k in range(3):
                c[:, k] = P[k, 0] * x + P[k, 1] * y + P[k, 2] * z + P[k, 3]
        out[b] = voxelize_points(c, volume_size, cuboid_side)
    return out

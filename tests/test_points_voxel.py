"""Point-cloud entry into the scene occupancy grid: point_cloud_to_voxel_numpy (network/voxel_net_depth.py:207-222),
point_cloud_to_voxel_pytorch (dataset/real_depth_utils.py:45-60) and the batched scatter sceneego_voxelize_points.
CPU: the point-cloud oracle (tests/points_oracle.py) pinned to the reference-generated depth goldens, its dtype rule,
argument checks.  GPU: bit-exact against the goldens and the oracle, ragged batches, the scene_volumes= path end to end,
both storage builds."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import sceneego_oracle as orc
from sceneego_b200 import _lib
from sceneego_b200.utils import synth
from tests import points_oracle as pto
from tests import util

NAMES = ("img_001000", "img_001796", "img_002376")


@pytest.fixture(scope="module")
def ray():
    return orc.ray_table(orc.load_calibration(util.CALIB), 1280, 1024)      # (W*H, 3) fp64, x-major


def _network_depth(d):
    """The map the network multiplies by its rays (voxel_net_depth.py:197-198): nearest squash to 1024 x 1024, 128
    zero columns each side."""
    d = orc.resize_nearest(np.asarray(d, np.float32), 1024, 1024)
    return np.pad(d, ((0, 0), (128, 128)), "constant", constant_values=0)


def _cloud(ray, d):
    """ray * depth, pixel for pixel, fp64 (voxel_net_depth.py:199-201, dataset/real_depth_utils.py:31-33)."""
    return (ray.T * d.T.reshape(-1)).T


# ---------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("V", [64, 128])
def test_oracle_points_equal_depth_goldens(ray, V):
    """voxelize_points of the clouds the network and the dataset build from the demo depth maps equals voxelize_depth
    / voxelize_depth_dataset and the occupancy the unmodified reference produced (tests/golden/voxel*.npz)."""
    g, gd = util.golden("voxel.npz"), util.golden("voxel_dataset.npz")
    for name in NAMES:
        d = orc.preprocess_depth(g[f"{name}_raw"])
        net = pto.voxelize_points(_cloud(ray, _network_depth(d)), V, 2.0)
        assert np.array_equal(net, orc.voxelize_depth(d, ray, V, 2.0)), name
        assert np.array_equal(net, util.unpack_bits(g[f"{name}_v{V}"], V)), name
        if name != "img_001796":                                   # the dataset golden holds the other two frames
            ds = pto.voxelize_points(_cloud(ray, d), V, 2.0)
            assert np.array_equal(ds, orc.voxelize_depth_dataset(d, ray, V, 2.0)), name
            assert np.array_equal(ds, util.unpack_bits(gd[f"{name}_v{V}"], V)), name


def _tie_cloud(V, s, dtype):
    """Points within a few ulps of every rounding tie q = k + 0.5 on each axis, in `dtype`."""
    k = np.arange(-1, V + 1, dtype=np.float64) + 0.5
    xy = (k * s / V - s / 2).astype(dtype)
    z = (k * s / V).astype(dtype)
    pts = []
    for steps in range(-6, 7):
        px = xy.copy()
        pz = z.copy()
        for _ in range(abs(steps)):
            px = np.nextafter(px, np.array(np.inf if steps > 0 else -np.inf, dtype))
            pz = np.nextafter(pz, np.array(np.inf if steps > 0 else -np.inf, dtype))
        mid_xy, mid_z = dtype(0.25), dtype(s / 4)
        n = px.shape[0]
        pts += [np.stack([px, np.full(n, mid_xy, dtype), np.full(n, mid_z, dtype)], 1),
                np.stack([np.full(n, mid_xy, dtype), px, np.full(n, mid_z, dtype)], 1),
                np.stack([np.full(n, mid_xy, dtype), np.full(n, mid_xy, dtype), pz], 1)]
    return np.concatenate(pts).astype(dtype)


def test_oracle_float32_cloud_is_computed_in_float32():
    """The dtype rule is real: the same float32 values quantised in fp32 and in fp64 land in different voxels, and the
    fp32 result is what float32 scalar arithmetic gives point by point."""
    for s in (2.5, 2.0, 1.7):
        p32 = _tie_cloud(64, s, np.float32)
        a = pto.voxelize_points(p32, 64, s)
        b = pto.voxelize_points(p32.astype(np.float64), 64, s)
        if s != 2.0:                                        # s = 2: (p + 1) * 32 is exact in fp32 for these points
            assert not np.array_equal(a, b), s
        f = np.float32
        want = np.zeros((64, 64, 64), np.float32)
        for x, y, z in p32[::7]:
            q = [np.round((x + f(s / 2)) * f(64) / f(s)), np.round((y + f(s / 2)) * f(64) / f(s)), np.round(z * f(64) / f(s))]
            assert all(isinstance(t, np.float32) for t in q)
            if all(0 <= t <= 63 for t in q):
                want[int(q[0]), int(q[1]), int(q[2])] = 1.0
        assert np.array_equal(pto.voxelize_points(p32[::7], 64, s), want), s


def test_voxelize_points_argument_checks():
    """_lib.voxelize_points rejects bad dtypes and shapes before touching a device; the C entry point rejects
    V <= 0, cuboid_side <= 0, batch < 0 and null pointers with SCENEEGO_E_INVALID, and batch == 0 is a no-op."""
    occ = torch.zeros(1, 8, 8, 8)
    off = torch.tensor([0, 4])
    for bad in (torch.zeros(4, 3, dtype=torch.float16), torch.zeros(4, 3, dtype=torch.int64), np.zeros((4, 3))):
        with pytest.raises(_lib.SceneEgoError, match="float64 or float32"):
            _lib.voxelize_points(bad, off, 8, 2.0, occ)
    for bad in (torch.zeros(4, 2, dtype=torch.float64), torch.zeros(12, dtype=torch.float64),
                torch.zeros(2, 2, 3, dtype=torch.float32)):
        with pytest.raises(_lib.SceneEgoError, match=r"shape \(N, 3\)"):
            _lib.voxelize_points(bad, off, 8, 2.0, occ)
    for bad in (torch.tensor([0, 4], dtype=torch.int32), torch.tensor([[0, 4]]), torch.zeros(0, dtype=torch.int64)):
        with pytest.raises(_lib.SceneEgoError, match="offsets"):
            _lib.voxelize_points(torch.zeros(4, 3, dtype=torch.float64), bad, 8, 2.0, occ)
    with pytest.raises(_lib.SceneEgoError, match="CUDA"):
        _lib.voxelize_points(torch.zeros(4, 3, dtype=torch.float64), off, 8, 2.0, occ)
    lib = _lib.load_library()
    f = lib.sceneego_voxelize_points
    dummy = C.c_void_p(0x1000)                            # never dereferenced: every case fails before a launch
    for args in ((dummy, 1, dummy, 1, 0, 2.0), (dummy, 1, dummy, 1, -4, 2.0), (dummy, 1, dummy, 1, 64, 0.0),
                 (dummy, 1, dummy, 1, 64, -2.0), (dummy, 1, dummy, 1, 64, float("nan")), (dummy, 1, dummy, -1, 64, 2.0),
                 (None, 1, dummy, 1, 64, 2.0), (dummy, 0, None, 1, 64, 2.0)):
        occ_p = dummy
        assert f(args[0], args[1], args[2], args[3], args[4], C.c_double(args[5]), occ_p, None) == -1, args
    assert f(dummy, 1, dummy, 1, 64, C.c_double(2.0), None, None) == -1
    assert b"voxelize_points" in lib.sceneego_last_error()
    assert f(dummy, 1, dummy, 0, 64, C.c_double(2.0), dummy, None) == 0       # batch 0: nothing launched


# ---------------------------------------------------------------------------------------------------------- GPU
def _gpu(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("V", [64, 128])
def test_depth_derived_clouds_bit_exact(ray, V):
    """The network's and the dataset's clouds of the demo frames, fp64, one batched call each: the occupancy the
    unmodified reference produced, bit for bit."""
    from sceneego_b200.dataset import real_depth_utils as rdu
    g, gd = util.golden("voxel.npz"), util.golden("voxel_dataset.npz")
    maps = [orc.preprocess_depth(g[f"{n}_raw"]) for n in NAMES]
    occ = rdu.point_clouds_to_voxels([_gpu(_cloud(ray, _network_depth(d))) for d in maps], None, 2.0, V)
    assert occ.shape == (3, V, V, V) and occ.dtype == torch.float32
    for i, n in enumerate(NAMES):
        assert torch.equal(occ[i], _gpu(util.unpack_bits(g[f"{n}_v{V}"], V))), n
    for i, n in ((0, "img_001000"), (2, "img_002376")):
        vox = rdu.point_cloud_to_voxel_pytorch(_gpu(_cloud(ray, maps[i])), 2.0, V)
        assert torch.equal(vox, _gpu(util.unpack_bits(gd[f"{n}_v{V}"], V))), n


def _planted(V, s, dtype):
    f = np.finfo(dtype)
    big = [f.max, f.max / 4, 1e30, -1e30, 3e38 if dtype == np.float32 else 1e300]
    faces = []
    for q in (-0.5, V - 0.5, V - 1.5, 0.0, V - 1.0):       # kept / dropped at each face, both sides of the tie
        for axis in range(3):
            base = np.array([0.1, -0.1, s / 4], np.float64)
            base[axis] = q * s / V - (s / 2 if axis < 2 else 0.0)
            p = base.astype(dtype)
            for d in (-np.inf, np.inf):
                faces.append(p.copy())
                t = p.copy()
                t[axis] = np.nextafter(t[axis], np.array(d, dtype))
                faces.append(t)
    weird = [[np.nan, 0, 0], [0, np.nan, 0], [0, 0, np.nan], [np.inf, 0, 0], [-np.inf, 0, 0], [0, np.inf, 0],
             [0, 0, -np.inf], [0, 0, np.inf], [-0.0, -0.0, -0.0], [0.0, 0.0, 0.0]]
    weird += [[b, 0, 0.5] for b in big] + [[0, b, 0.5] for b in big] + [[0, 0, b] for b in big]
    rng = np.random.default_rng(int(V * 10 + s * 100))
    rnd = (rng.random((20000, 3)) * 1.4 - 0.2) * np.array([s, s, s]) - np.array([s / 2, s / 2, 0.0])
    return np.concatenate([_tie_cloud(V, s, dtype), np.array(faces, dtype), np.array(weird, dtype),
                           rnd.astype(dtype)]).astype(dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_planted_edge_cases_vs_oracle(dtype):
    """Exact rounding ties, q = -0.5 (-0.0, kept), q = V - 0.5 (rounds to V, dropped), one ulp inside / outside every
    face, NaN / inf / huge points; power-of-two and other sides and volume sizes (all three quantisation paths)."""
    from sceneego_b200.dataset import real_depth_utils as rdu
    for V, s in ((64, 2.0), (64, 4.0), (64, 2.5), (48, 2.0), (48, 2.5), (64, 1.7)):
        pts = _planted(V, s, dtype)
        with np.errstate(all="ignore"):
            want = pto.voxelize_points(pts, V, s)
        got = rdu.point_cloud_to_voxel_pytorch(_gpu(pts), s, V)
        assert torch.equal(got.cpu(), torch.from_numpy(want)), (V, s)
        assert want.sum() > 100, (V, s)
    # q = -0.5 -> -0.0 is kept, q = V - 0.5 -> V is dropped
    s, V = 2.0, 64
    p = np.array([[-0.5 / 32 - 1, 0.0, 0.5], [63.5 / 32 - 1, 0.0, 0.5], [0.0, 0.0, -0.5 / 32], [0.0, 0.0, 63.5 / 32]],
                 dtype)
    got = rdu.point_clouds_to_voxels(_gpu(p), [1, 1, 1, 1], s, V).cpu().numpy()
    assert got[0, 0, 32, 16] == 1.0 and got[0].sum() == 1
    assert got[1].sum() == 0 and got[3].sum() == 0
    assert got[2, 32, 32, 0] == 1.0 and got[2].sum() == 1


@pytest.mark.gpu
def test_ragged_batches_equal_single_frame_calls(ray):
    """B = 1, B = 7 with an empty frame (offsets and counts, tensor and list inputs), and B = 64 at 1.31 M points per
    frame (synthetic room clouds): every frame of the batch equals the frame alone; the row-major ray x depth cloud
    equals the dataset voxelisation of the same maps (another kernel)."""
    from sceneego_b200.dataset import real_depth_utils as rdu
    rng = np.random.default_rng(5)
    clouds = [(rng.random((n, 3)) * 2.4 - np.array([1.2, 1.2, 0.1])) for n in (5000, 1, 77777, 0, 4096, 123, 31)]
    single = [rdu.point_cloud_to_voxel_pytorch(_gpu(c), 2.0, 64) for c in clouds]
    assert single[3].sum().item() == 0
    flat = _gpu(np.concatenate(clouds))
    counts = [c.shape[0] for c in clouds]
    offsets = np.concatenate([[0], np.cumsum(counts)])
    for batch in (rdu.point_clouds_to_voxels(flat, counts, 2.0, 64),
                  rdu.point_clouds_to_voxels(flat, torch.from_numpy(offsets).cuda(), 2.0, 64),
                  rdu.point_clouds_to_voxels([_gpu(c) for c in clouds], None, 2.0, 64)):
        assert batch.shape[0] == 7
        for i in range(7):
            assert torch.equal(batch[i], single[i]), i
    one = rdu.point_clouds_to_voxels(_gpu(clouds[0]), [counts[0]], 2.0, 64)
    assert one.shape[0] == 1 and torch.equal(one[0], single[0])
    for bad in ([1, 2], [0, 5, 3, flat.shape[0]], [-1, flat.shape[0] + 1]):
        with pytest.raises(_lib.SceneEgoError):
            rdu.point_clouds_to_voxels(flat, bad, 2.0, 64)
    # B = 64, 1.31 M points per frame, fp64
    from sceneego_b200.utils.fisheye.FishEyeCalibrated import FishEyeCameraCalibrated
    ray_dev = FishEyeCameraCalibrated(util.CALIB).ray_table_device(1280, 1024, "cuda")
    depth = synth.synthetic_depth_room(64, ray, seed=21).cuda()
    pts = (ray_dev.unsqueeze(0) * depth.double().unsqueeze(-1)).reshape(-1, 3)
    occ = rdu.point_clouds_to_voxels(pts, [1024 * 1280] * 64, 2.0, 64)
    assert torch.equal(occ, rdu.depth_maps_to_voxels(ray_dev, depth, 2.0, 64, preprocess=False))
    for i in (0, 17, 63):
        assert torch.equal(occ[i], rdu.point_cloud_to_voxel_pytorch(pts[i * 1310720:(i + 1) * 1310720], 2.0, 64)), i
    assert torch.equal(occ[40].cpu(), torch.from_numpy(pto.voxelize_points(pts[40 * 1310720:41 * 1310720].cpu().numpy(),
                                                                           64, 2.0)))
    occ32 = rdu.point_clouds_to_voxels(pts.float(), [1024 * 1280] * 64, 2.0, 64)
    assert torch.equal(occ32[9].cpu(), torch.from_numpy(pto.voxelize_points(pts[9 * 1310720:10 * 1310720].float().cpu()
                                                                             .numpy(), 64, 2.0)))


@pytest.fixture(scope="module")
def net():
    from sceneego_b200.network.voxel_net_depth import VoxelNetwork_depth
    torch.manual_seed(0)
    n = VoxelNetwork_depth(util.load_config(batch_size=4), device="cuda").eval()
    sd = synth.synthetic_state_dict(util.stage_shapes(), seed=0, mode="random_bn")
    full = n.state_dict()
    full.update(sd)
    n.load_state_dict(full, strict=True)
    return n


@pytest.mark.gpu
def test_lift_with_point_cloud_scene_equals_depth_path(net, ray):
    """lift(scene_volumes=stack of point_cloud_to_voxel_numpy(cloud_b)) with the network's own ray x depth clouds
    gives the keypoints of lift(depth_map_batch=...), bit for bit."""
    depth = torch.cat([synth.synthetic_depth_room(2, ray, seed=31), synth.synthetic_depth_uniform(1, seed=32)])
    feat = synth.synthetic_features(3, seed=33).cuda()
    ray_dev = net._ray_dev                                                # (1024, 1280, 3) fp64, row-major
    cols = torch.from_numpy(orc.nearest_index(1280, 1024)).cuda()
    grids = []
    for d in depth.cuda():
        sq = torch.nn.functional.pad(d[:, cols], (128, 128))            # squash to 1024 x 1024, pad (:197-198)
        cloud = (ray_dev * sq.double().unsqueeze(-1)).reshape(-1, 3)
        grids.append(net.point_cloud_to_voxel_numpy(cloud))
        assert torch.equal(grids[-1], net.depth_map_to_voxel_numpy(d))
    sv = torch.stack(grids)
    with torch.no_grad():
        a = net.lift(feat, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=depth.cuda())[0]
        b = net.lift(feat, net.grid_coord_proj_batch, net.coord_volumes, scene_volumes=sv)[0]
    assert torch.equal(a, b)


@pytest.mark.gpu
def test_module_point_cloud_and_ray_api(net, ray):
    """calculated_ray_direction_numpy(1280, 1024) is the module's x-major fp64 `ray`; point_cloud_to_voxel_numpy takes
    NumPy arrays and CPU / CUDA tensors alike (the result lives on the module's device) and keeps the cloud's dtype."""
    r = net.calculated_ray_direction_numpy(1280, 1024)
    assert isinstance(r, np.ndarray) and r.dtype == np.float64 and r.shape == (1280 * 1024, 3)
    assert np.array_equal(r, net.ray) and np.array_equal(r, ray)
    small = net.calculated_ray_direction_numpy(64, 48)
    assert small.shape == (64 * 48, 3) and np.array_equal(small, orc.ray_table(orc.load_calibration(util.CALIB), 64, 48))
    d = synth.synthetic_depth_room(1, ray, seed=41)[0].numpy()
    cloud = _cloud(ray, d)
    a = net.point_cloud_to_voxel_numpy(cloud)
    assert a.is_cuda and a.shape == (64, 64, 64) and a.dtype == torch.float32
    for other in (torch.from_numpy(cloud), torch.from_numpy(cloud).cuda()):
        assert torch.equal(net.point_cloud_to_voxel_numpy(other), a)
    assert torch.equal(a.cpu(), torch.from_numpy(pto.voxelize_points(cloud, 64, 2.0)))
    c32 = _planted(64, 2.5, np.float32)
    side = net.cuboid_side
    net.cuboid_side = 2.5
    try:
        with np.errstate(all="ignore"):
            want = pto.voxelize_points(c32, 64, 2.5)
        assert torch.equal(net.point_cloud_to_voxel_numpy(c32).cpu(), torch.from_numpy(want))
    finally:
        net.cuboid_side = side
    with pytest.raises(_lib.SceneEgoError):
        net.point_cloud_to_voxel_numpy(cloud.astype(np.float16))


@pytest.mark.gpu
@pytest.mark.skipif(os.environ.get("SCENEEGO_ACT_DTYPE", "bf16").lower() in ("f16", "fp16", "float16"),
                    reason="already running on the fp16-storage build")
def test_points_voxel_with_fp16_storage_build():
    """This file's GPU tests on libsceneego_b200_f16.so (one activation dtype per process: a subprocess)."""
    env = dict(os.environ, SCENEEGO_ACT_DTYPE="f16", PYTHONPATH=util.ROOT)
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_points_voxel.py", "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider"], cwd=util.ROOT, env=env, capture_output=True, text=True, timeout=1200)
    tail = (r.stdout + r.stderr)[-1500:]
    assert r.returncode == 0, tail
    assert " passed" in tail.splitlines()[-1]

"""Scene occupancy from one world-space scan and per-frame camera poses: sceneego_voxelize_scan,
real_depth_utils.scan_to_voxels and VoxelNetwork_depth.scan_to_voxels.
CPU: the scan restatement (tests/scan_oracle.voxelize_scan) tied to voxelize_points and, through signed-permutation
poses, to the reference-generated depth goldens; its dtype rule; argument checks of the binding and the C entry point.
GPU: bit-exact against the restatement (rigid and affine poses, all three quantisation paths, planted edge cases),
against voxelize_points of the transformed clouds, the goldens, the scene_volumes= path end to end, both storage
builds."""
import ctypes as C
import itertools
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
from tests import scan_oracle as sco
from tests import util
from tests.test_points_voxel import NAMES, _cloud, _network_depth, _planted, _tie_cloud

PLANTED_VS = ((64, 2.0), (64, 4.0), (64, 2.5), (48, 2.5), (128, 2.0))


def _signed_perms():
    """All 48 signed 3x3 permutation matrices (fp64)."""
    out = []
    for perm in itertools.permutations(range(3)):
        for signs in itertools.product((1.0, -1.0), repeat=3):
            P = np.zeros((3, 3))
            for r, c in enumerate(perm):
                P[r, c] = signs[r]
            out.append(P)
    return out


def _pose(A, t=(0.0, 0.0, 0.0), dtype=np.float64):
    M = np.eye(4)
    M[:3, :3], M[:3, 3] = A, t
    return M.astype(dtype)


def _to_world(cam, P):
    """world = P . cam for a signed permutation P, exactly: each world coordinate is +-one camera coordinate."""
    out = np.empty_like(cam)
    for r in range(3):
        c = int(np.flatnonzero(P[r])[0])
        out[:, r] = cam[:, c] if P[r, c] > 0 else -cam[:, c]
    return out


def _random_poses(B, rng, affine, dtype, spread=0.3):
    """Rigid poses (random rotation, translation of a few cm) or affine ones (random 3x3 near the identity)."""
    out = np.zeros((B, 4, 4))
    for b in range(B):
        if affine:
            A = np.eye(3) + rng.normal(0, spread, (3, 3))
        else:
            q, r = np.linalg.qr(rng.normal(size=(3, 3)))
            A = q * np.sign(np.diag(r))
            if np.linalg.det(A) < 0:
                A[:, 0] = -A[:, 0]
        out[b] = _pose(A, rng.normal(0, 0.05, 3))
    return out.astype(dtype)


@pytest.fixture(scope="module")
def ray():
    return orc.ray_table(orc.load_calibration(util.CALIB), 1280, 1024)      # (W*H, 3) fp64, x-major


# ---------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_oracle_identity_pose_equals_voxelize_points(dtype):
    """An identity pose gives voxelize_points of the scan itself (only the sign of a zero can differ, which no index
    sees), planted edge cases included."""
    for V, s in ((64, 2.0), (48, 2.5)):
        pts = _planted(V, s, dtype)
        with np.errstate(all="ignore"):
            want = pto.voxelize_points(pts, V, s)
            got = sco.voxelize_scan(pts, _pose(np.eye(3), dtype=dtype)[None], V, s)
        assert got.shape == (1, V, V, V) and np.array_equal(got[0], want), (V, s)


@pytest.mark.parametrize("V", [64, 128])
def test_oracle_permuted_demo_clouds_equal_goldens(ray, V):
    """The network's clouds of the demo frames carried to world space by signed permutations (world = P cam, exact)
    and brought back with cam_from_world = P^T reproduce the occupancy the unmodified reference produced."""
    g = util.golden("voxel.npz")
    perms = _signed_perms()
    for i, name in enumerate(NAMES):
        cam = _cloud(ray, _network_depth(orc.preprocess_depth(g[f"{name}_raw"])))
        P = perms[(7 * i + 5) % len(perms)]
        got = sco.voxelize_scan(_to_world(cam, P), _pose(P.T)[None], V, 2.0)[0]
        assert np.array_equal(got, util.unpack_bits(g[f"{name}_v{V}"], V)), name


def test_oracle_float32_scan_is_transformed_in_float32():
    """fp32 scans and poses are transformed and quantised in fp32: the result is what float32 scalar arithmetic
    gives point by point, and differs from the fp64 computation of the same values."""
    rng = np.random.default_rng(3)
    f = np.float32
    cam = _tie_cloud(64, 2.5, np.float64)
    pose = _random_poses(1, rng, affine=False, dtype=np.float64)[0]
    world = ((cam - pose[:3, 3]) @ pose[:3, :3]).astype(f)              # inverse of a rigid pose, then rounded to f32
    p32 = pose.astype(f)
    a = sco.voxelize_scan(world, p32[None], 64, 2.5)[0]
    b = sco.voxelize_scan(world.astype(np.float64), p32.astype(np.float64)[None], 64, 2.5)[0]
    assert not np.array_equal(a, b)
    want = np.zeros((64, 64, 64), np.float32)
    for x, y, z in world[::5]:
        c = [p32[k, 0] * x + p32[k, 1] * y + p32[k, 2] * z + p32[k, 3] for k in range(3)]
        q = [np.round((c[0] + f(1.25)) * f(64) / f(2.5)), np.round((c[1] + f(1.25)) * f(64) / f(2.5)),
             np.round(c[2] * f(64) / f(2.5))]
        assert all(isinstance(t, np.float32) for t in c + q)
        if all(0 <= t <= 63 for t in q):
            want[int(q[0]), int(q[1]), int(q[2])] = 1.0
    assert np.array_equal(sco.voxelize_scan(world[::5], p32[None], 64, 2.5)[0], want)


def test_voxelize_scan_argument_checks():
    """_lib.voxelize_scan rejects bad dtypes, shapes, a pose dtype that differs from the scan's, non-finite poses, a
    bottom row other than (0,0,0,1), a wrong occupancy buffer and a CPU scan before touching a device; the C entry
    point rejects null pointers and out-of-range sizes with SCENEEGO_E_INVALID and sets sceneego_last_error."""
    occ = torch.zeros(2, 8, 8, 8)
    scan = torch.zeros(4, 3, dtype=torch.float64)
    pose = torch.eye(4, dtype=torch.float64).repeat(2, 1, 1)
    for bad in (torch.zeros(4, 3, dtype=torch.float16), torch.zeros(4, 3, dtype=torch.int64), np.zeros((4, 3))):
        with pytest.raises(_lib.SceneEgoError, match="float64 or float32"):
            _lib.voxelize_scan(bad, pose, 8, 2.0, occ)
    for bad in (torch.zeros(4, 2, dtype=torch.float64), torch.zeros(12, dtype=torch.float64),
                torch.zeros(2, 2, 3, dtype=torch.float64)):
        with pytest.raises(_lib.SceneEgoError, match=r"shape \(N, 3\)"):
            _lib.voxelize_scan(bad, pose, 8, 2.0, occ)
    for bad in (torch.eye(4, dtype=torch.float64), torch.zeros(2, 3, 4, dtype=torch.float64),
                torch.zeros(2, 4, 3, dtype=torch.float64), np.eye(4)[None].repeat(2, 0)):
        with pytest.raises(_lib.SceneEgoError, match=r"\(B, 4, 4\)"):
            _lib.voxelize_scan(scan, bad, 8, 2.0, occ)
    with pytest.raises(_lib.SceneEgoError, match="dtype"):
        _lib.voxelize_scan(scan, pose.float(), 8, 2.0, occ)
    with pytest.raises(_lib.SceneEgoError, match="dtype"):
        _lib.voxelize_scan(scan.float(), pose, 8, 2.0, occ)
    for v in (float("nan"), float("inf"), -float("inf")):
        bad = pose.clone()
        bad[1, 0, 2] = v
        with pytest.raises(_lib.SceneEgoError, match="non-finite"):
            _lib.voxelize_scan(scan, bad, 8, 2.0, occ)
    for idx, v in (((0, 3, 0), 1e-300), ((1, 3, 3), 2.0), ((0, 3, 2), -0.5), ((1, 3, 3), 1.0 + 2 ** -52)):
        bad = pose.clone()
        bad[idx] = v
        with pytest.raises(_lib.SceneEgoError, match="bottom row"):
            _lib.voxelize_scan(scan, bad, 8, 2.0, occ)
    for bad in (torch.zeros(2, 8, 8, 8, dtype=torch.float64), torch.zeros(3, 8, 8, 8), torch.zeros(2, 8, 8, 4),
                torch.zeros(2, 512), None):
        with pytest.raises(_lib.SceneEgoError, match="occ_f32"):
            _lib.voxelize_scan(scan, pose, 8, 2.0, bad)
    with pytest.raises(_lib.SceneEgoError, match="CUDA"):
        _lib.voxelize_scan(scan, pose, 8, 2.0, occ)
    lib = _lib.load_library()
    f = lib.sceneego_voxelize_scan
    dummy = C.c_void_p(0x1000)                            # never dereferenced: every case fails before a launch
    good = (dummy, 1, 4, dummy, 2, 64, 2.0, dummy)
    bads = [(0, None), (3, None), (7, None), (5, 0), (5, -4), (5, 4097), (6, 0.0), (6, -2.0), (6, float("nan")),
            (4, -1), (2, -1), (4, 65535 * 32 + 1), (2, 2 ** 62)]
    for i, v in bads:
        args = list(good)
        args[i] = v
        rc = f(args[0], args[1], C.c_int64(args[2]), args[3], args[4], args[5], C.c_double(args[6]), args[7], None)
        assert rc == -1, (i, v)
        assert b"voxelize_scan" in lib.sceneego_last_error()
    for i, v in ((4, 0), (2, 0)):                         # batch 0 / no points: nothing launched
        args = list(good)
        args[i] = v
        assert f(args[0], args[1], C.c_int64(args[2]), args[3], args[4], args[5], C.c_double(args[6]), args[7],
                 None) == 0, (i, v)


# ---------------------------------------------------------------------------------------------------------- GPU
def _gpu(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _rdu():
    from sceneego_b200.dataset import real_depth_utils as rdu
    return rdu


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("affine", [False, True])
def test_random_poses_vs_oracle(dtype, affine):
    """Rigid and affine poses, fp32 and fp64, power-of-two and other sides and volume sizes (all three quantisation
    paths), on a synthetic room scan with a planted cloud carried into the cuboid's neighbourhood."""
    rng = np.random.default_rng(11 + affine)
    for V, s in PLANTED_VS:
        # the room scaled and centred on the camera, so that every pose sees part of it, plus the planted cloud
        scan = (synth.synthetic_world_scan(60000, seed=V, dtype=np.float64) - np.array([5.0, 4.0, 0.0])) * (s / 4)
        scan = np.concatenate([scan.astype(dtype), _planted(V, s, dtype)])
        poses = _random_poses(5, rng, affine, dtype)
        want = sco.voxelize_scan(scan, poses, V, s)
        got = _rdu().scan_to_voxels(_gpu(scan), poses, s, V)
        assert got.shape == (5, V, V, V) and got.dtype == torch.float32
        assert torch.equal(got.cpu(), torch.from_numpy(want)), (V, s)
        assert want.reshape(5, -1).sum(1).min() > 50, (V, s)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_planted_edge_cases_carried_by_signed_permutations(dtype):
    """Rounding ties, faces +-1 ulp, NaN / inf / huge points of test_points_voxel's planted clouds, carried to world
    space by signed permutations (exact) and brought back by the transposed poses: the restatement, voxelize_points
    of the camera-space cloud, and the kernel agree bit for bit, on every quantisation path."""
    perms = _signed_perms()
    for j, (V, s) in enumerate(PLANTED_VS):
        cam = _planted(V, s, dtype)
        with np.errstate(all="ignore"):
            base = pto.voxelize_points(cam, V, s)
        for P in perms[j::9]:
            world = _to_world(cam, P)
            poses = np.stack([_pose(P.T, dtype=dtype), _pose(np.eye(3), dtype=dtype)])
            want = sco.voxelize_scan(world, poses, V, s)
            assert np.array_equal(want[0], base), (V, s)
            got = _rdu().scan_to_voxels(_gpu(world), _gpu(poses), s, V).cpu()
            assert torch.equal(got, torch.from_numpy(want)), (V, s, P.tolist())
        assert base.sum() > 100


@pytest.mark.gpu
def test_identity_pose_equals_point_clouds_to_voxels():
    rdu = _rdu()
    rng = np.random.default_rng(4)
    for dtype in (np.float64, np.float32):
        cloud = _gpu((rng.random((300000, 3)) * 2.4 - np.array([1.2, 1.2, 0.1])).astype(dtype))
        want = rdu.point_clouds_to_voxels(cloud, [cloud.shape[0]], 2.0, 64)
        got = rdu.scan_to_voxels(cloud, torch.eye(4, dtype=cloud.dtype).repeat(3, 1, 1), 2.0, 64)
        for b in range(3):
            assert torch.equal(got[b], want[0]), (dtype, b)


@pytest.mark.gpu
@pytest.mark.parametrize("V", [64, 128])
def test_permuted_demo_clouds_equal_goldens(ray, V):
    """The three demo frames' network clouds, each carried to world space by its own signed permutation, in one call
    on the same world scan: frame i with pose P_i^T reproduces demo frame i's golden where it comes from scan i."""
    g = util.golden("voxel.npz")
    perms = _signed_perms()
    for i, name in enumerate(NAMES):
        cam = _cloud(ray, _network_depth(orc.preprocess_depth(g[f"{name}_raw"])))
        Ps = [perms[(7 * i + 5 + 13 * k) % len(perms)] for k in range(2)]
        world = _gpu(_to_world(cam, Ps[0]))
        got = _rdu().scan_to_voxels(world, np.stack([_pose(P.T) for P in Ps]), 2.0, V)
        assert torch.equal(got[0], _gpu(util.unpack_bits(g[f"{name}_v{V}"], V))), name
        other = sco.voxelize_scan(_to_world(cam, Ps[0]), _pose(Ps[1].T)[None], V, 2.0)[0]
        assert torch.equal(got[1].cpu(), torch.from_numpy(other)), name


def _torch_route(scan, poses, V, s):
    """What a user writes without sceneego_voxelize_scan: each frame's cloud in torch, A[k,0]*x + A[k,1]*y +
    A[k,2]*z + t[k] elementwise (the same operation order), then voxelize_points frame by frame."""
    rdu = _rdu()
    out = []
    x, y, z = scan[:, 0], scan[:, 1], scan[:, 2]
    for P in poses:
        cam = torch.stack([P[k, 0] * x + P[k, 1] * y + P[k, 2] * z + P[k, 3] for k in range(3)], 1)
        out.append(rdu.point_clouds_to_voxels(cam, [cam.shape[0]], s, V)[0])
    return torch.stack(out)


@pytest.mark.gpu
def test_batch64_multi_million_scan_equals_transformed_clouds():
    """B = 64 head poses over a 3 M-point room scan (two frame tiles), fp64 and fp32: every grid equals voxelize_points
    of the torch-transformed cloud; two frames against the NumPy restatement."""
    rdu = _rdu()
    for dtype in (np.float64, np.float32):
        scan_np = synth.synthetic_world_scan(3_000_000, seed=5, dtype=dtype)
        poses_np = synth.synthetic_head_trajectory(64, seed=6, dtype=dtype)
        scan, poses = _gpu(scan_np), _gpu(poses_np)
        got = rdu.scan_to_voxels(scan, poses, 2.0, 64)
        assert got.shape == (64, 64, 64, 64)
        assert torch.equal(got, _torch_route(scan, poses, 64, 2.0)), dtype
        for b in (0, 45):
            assert torch.equal(got[b].cpu(), torch.from_numpy(sco.voxelize_scan(scan_np, poses_np[b:b + 1], 64, 2.0)[0]))
        assert got.reshape(64, -1).sum(1).min() > 500


@pytest.mark.gpu
def test_batch_edge_cases():
    """B = 1; B = 0 and N = 0 give empty results without a launch; a frame whose cuboid sees nothing is all zero;
    repeated identical poses give identical grids; B = 70 (three frame tiles, the last partial) equals the
    restatement frame for frame."""
    rdu = _rdu()
    scan_np = synth.synthetic_world_scan(200000, seed=8)
    scan = _gpu(scan_np)
    poses = synth.synthetic_head_trajectory(70, seed=9)
    one = rdu.scan_to_voxels(scan, poses[:1], 2.0, 64)
    assert one.shape == (1, 64, 64, 64) and torch.equal(one[0].cpu(), torch.from_numpy(sco.voxelize_scan(
        scan_np, poses[:1], 64, 2.0)[0]))
    assert rdu.scan_to_voxels(scan, np.zeros((0, 4, 4)), 2.0, 64).shape == (0, 64, 64, 64)
    empty = rdu.scan_to_voxels(_gpu(np.zeros((0, 3))), poses[:3], 2.0, 64)
    assert empty.shape == (3, 64, 64, 64) and empty.sum().item() == 0
    away = poses[:2].copy()
    away[1, :3, 3] += np.array([0.0, 0.0, -50.0])             # the cuboid 50 m behind the camera: nothing in it
    got = rdu.scan_to_voxels(scan, away, 2.0, 64)
    assert got[0].sum().item() > 0 and got[1].sum().item() == 0
    rep = np.repeat(poses[3:4], 40, axis=0)
    got = rdu.scan_to_voxels(scan, rep, 2.0, 64)
    assert all(torch.equal(got[b], got[0]) for b in range(40)) and got[0].sum().item() > 0
    got = rdu.scan_to_voxels(scan, poses, 2.5, 48)
    assert torch.equal(got.cpu(), torch.from_numpy(sco.voxelize_scan(scan_np, poses, 48, 2.5)))
    with pytest.raises(_lib.SceneEgoError, match="dtype"):
        rdu.scan_to_voxels(scan, poses.astype(np.float32), 2.0, 64)


def _make_net(**kw):
    from sceneego_b200.network.voxel_net_depth import VoxelNetwork_depth
    torch.manual_seed(0)
    n = VoxelNetwork_depth(util.load_config(batch_size=4), device="cuda", **kw).eval()
    sd = synth.synthetic_state_dict(util.stage_shapes(), seed=0, mode="random_bn")
    full = n.state_dict()
    full.update(sd)
    n.load_state_dict(full, strict=True)
    return n


@pytest.fixture(scope="module")
def net():
    return _make_net()


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_lift_with_scan_scene_equals_transformed_clouds(net, graph):
    """lift(scene_volumes=net.scan_to_voxels(scan, poses)) gives the keypoints of lift(scene_volumes=...) built from
    the per-frame transformed clouds with point_cloud_to_voxel_numpy, bit for bit, eager and as a CUDA graph
    (graph_max_batch)."""
    m = _make_net(graph_max_batch=4) if graph else net
    scan = _gpu(synth.synthetic_world_scan(1_000_000, seed=12))
    poses = _gpu(synth.synthetic_head_trajectory(3, seed=13))
    feat = synth.synthetic_features(3, seed=14).cuda()
    x, y, z = scan[:, 0], scan[:, 1], scan[:, 2]
    per_frame = torch.stack([m.point_cloud_to_voxel_numpy(torch.stack(
        [P[k, 0] * x + P[k, 1] * y + P[k, 2] * z + P[k, 3] for k in range(3)], 1)) for P in poses])
    sv = m.scan_to_voxels(scan, poses)
    assert torch.equal(sv, per_frame) and sv.sum().item() > 0
    with torch.no_grad():
        a = m.lift(feat, m.grid_coord_proj_batch, m.coord_volumes, scene_volumes=per_frame)[0]
        b = m.lift(feat, m.grid_coord_proj_batch, m.coord_volumes, scene_volumes=sv)[0]
    assert torch.equal(a, b)
    if graph:
        assert len(m._graphs) == 1                          # both calls replayed the one scene_volumes capture
        with torch.no_grad():
            e = net.lift(feat, net.grid_coord_proj_batch, net.coord_volumes, scene_volumes=sv)[0]
        assert torch.equal(b, e)


@pytest.mark.gpu
def test_module_scan_api_accepts_numpy_cpu_and_cuda(net):
    """VoxelNetwork_depth.scan_to_voxels takes NumPy arrays and CPU / CUDA tensors for the scan and the poses, uses
    the module's volume_size and cuboid_side, and returns grids on the module's device."""
    scan = synth.synthetic_world_scan(100000, seed=15)
    poses = synth.synthetic_head_trajectory(4, seed=16)
    want = torch.from_numpy(sco.voxelize_scan(scan, poses, net.volume_size, net.cuboid_side))
    for s_in, p_in in ((scan, poses), (torch.from_numpy(scan), torch.from_numpy(poses)),
                       (_gpu(scan), _gpu(poses)), (torch.from_numpy(scan), _gpu(poses))):
        got = net.scan_to_voxels(s_in, p_in)
        assert got.is_cuda and got.shape == (4, 64, 64, 64) and got.dtype == torch.float32
        assert torch.equal(got.cpu(), want)
    s32, p32 = scan.astype(np.float32), poses.astype(np.float32)
    assert torch.equal(net.scan_to_voxels(s32, p32).cpu(),
                       torch.from_numpy(sco.voxelize_scan(s32, p32, net.volume_size, net.cuboid_side)))
    with pytest.raises(_lib.SceneEgoError):
        net.scan_to_voxels(scan.astype(np.float16), poses)


@pytest.mark.gpu
@pytest.mark.skipif(os.environ.get("SCENEEGO_ACT_DTYPE", "bf16").lower() in ("f16", "fp16", "float16"),
                    reason="already running on the fp16-storage build")
def test_scan_voxel_with_fp16_storage_build():
    """This file's GPU tests on libsceneego_b200_f16.so (one activation dtype per process: a subprocess)."""
    env = dict(os.environ, SCENEEGO_ACT_DTYPE="f16", PYTHONPATH=util.ROOT)
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_scan_voxel.py", "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider"], cwd=util.ROOT, env=env, capture_output=True, text=True, timeout=1200)
    tail = (r.stdout + r.stderr)[-1500:]
    assert r.returncode == 0, tail
    assert " passed" in tail.splitlines()[-1]

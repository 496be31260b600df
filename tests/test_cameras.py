"""A fisheye calibration per frame: `VoxelNetwork_depth.add_camera` and `camera_ids=`.

The specification: with camera k set up from calibration file f_k, frame b of
`net.lift(..., camera_ids=ids)` equals, bit for bit, frame b of a module built from f_{ids[b]} with the same state dict
lifting the same batch (keypoints, output #3, the V2V logits and output #2), on every input path and switch.  Kernel
tests compare the camera-per-frame gather with one `sceneego_unproject_f32` launch per camera on that camera's frames,
and the camera-per-frame voxelisation with the NumPy oracle run with each camera's ray table.  Destinations carry a
spare frame holding a sentinel (NaN, 0xFFFF for 16-bit volumes) that must stay untouched.  The GPU tests also run on
the fp16-storage build, in a subprocess."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import sceneego_oracle as orc
from sceneego_b200.utils import synth
from tests import util

F16_RUN = os.environ.get("SCENEEGO_ACT_DTYPE", "bf16").lower() in ("f16", "fp16", "float16")
IMG_H, IMG_W = 1024, 1280


# ---- calibrations ------------------------------------------------------------------------------------------------------
def _write_calib(path, shift=(0.0, 0.0), scale_c2w=1.0, scale_w2c=1.0, size=None):
    """The 05_08 calibration with the image centre shifted (the older file differs from it there) and/or the
    polynomial coefficients scaled."""
    d = json.load(open(util.CALIB))
    d["intrinsic"][0][2] += shift[0]
    d["intrinsic"][1][2] += shift[1]
    d["polynomialC2W"] = [c * scale_c2w for c in d["polynomialC2W"]]
    d["polynomialW2C"] = [c * scale_w2c for c in d["polynomialW2C"]]
    if size is not None:
        d["size"] = list(size)
    with open(path, "w") as f:
        json.dump(d, f)
    return str(path)


def _calib_variant(k):
    """Camera k of the kernel tests: 0 is 05_08, 1 a shifted centre, 2 scaled polynomials, then mixtures."""
    if k == 0:
        return dict()
    if k == 1:
        return dict(shift=(-7.25, 11.5))
    if k == 2:
        return dict(scale_c2w=1.03, scale_w2c=0.97)
    return dict(shift=(1.5 * k - 12.0, 9.0 - 1.25 * k), scale_c2w=1.0 + 0.004 * k, scale_w2c=1.0 - 0.003 * k)


@pytest.fixture(scope="module")
def calib_files(tmp_path_factory):
    d = tmp_path_factory.mktemp("calib")
    return [util.CALIB] + [_write_calib(d / f"cam{k}.json", **_calib_variant(k)) for k in range(1, 16)]


# ---- CPU: argument checks ---------------------------------------------------------------------------------------------
def test_add_camera_takes_a_path_or_a_model(calib_files):
    from sceneego_b200.network.voxel_net_depth import _camera_model
    from sceneego_b200.utils.fisheye.FishEyeCalibrated import FishEyeCameraCalibrated
    m = _camera_model(calib_files[1], (IMG_W, IMG_H), 1)
    assert m.img_center[0] == json.load(open(calib_files[1]))["intrinsic"][0][2]
    obj = FishEyeCameraCalibrated(calib_files[2])
    assert _camera_model(obj, (IMG_W, IMG_H), 15) is obj
    from sceneego_b200 import _lib
    with pytest.raises(_lib.SceneEgoError, match="file path or a FishEyeCameraCalibrated"):
        _camera_model(3, (IMG_W, IMG_H), 1)


def test_add_camera_refuses_another_image_size(tmp_path):
    from sceneego_b200 import _lib
    from sceneego_b200.network.voxel_net_depth import _camera_model
    small = _write_calib(tmp_path / "small.json", size=(640, 512))
    with pytest.raises(_lib.SceneEgoError, match="differs from the module's"):
        _camera_model(small, (IMG_W, IMG_H), 1)


def test_add_camera_refuses_a_17th_camera(calib_files):
    from sceneego_b200 import _lib
    from sceneego_b200.network.voxel_net_depth import _camera_model
    with pytest.raises(_lib.SceneEgoError, match="at most 16 cameras"):
        _camera_model(calib_files[1], (IMG_W, IMG_H), 16)


@pytest.mark.parametrize("bad,match", [
    ([0, 1], "one id per frame"),
    ([0, 1, 2, 0], "one id per frame"),
    ([0, 3, 1], r"lie in \[0, 3\)"),
    ([0, -1, 1], r"lie in \[0, 3\)"),
    ([0.0, 1.0, 2.0], "integers"),
    (np.array([0, 1, 2], np.float32), "integers"),
    (torch.tensor([0.0, 1.0, 2.0]), "integers"),
    (torch.tensor([True, False, True]), "integers"),
    (np.zeros((3, 1), np.int64), "one id per frame"),
    (torch.zeros(3, dtype=torch.int64, device="meta"), "host-side sequence"),
])
def test_camera_ids_are_checked_on_the_host(bad, match):
    from sceneego_b200 import _lib
    from sceneego_b200.network.voxel_net_depth import camera_ids_host
    with pytest.raises(_lib.SceneEgoError, match=match):
        camera_ids_host(bad, 3, 3)


@pytest.mark.parametrize("ok", [[2, 0, 1], np.array([2, 0, 1], np.uint8), torch.tensor([2, 0, 1], dtype=torch.int16)])
def test_camera_ids_accepted_forms(ok):
    from sceneego_b200.network.voxel_net_depth import camera_ids_host
    got = camera_ids_host(ok, 3, 3)
    assert got.dtype == np.int32 and got.tolist() == [2, 0, 1]


def test_frame_order_is_a_stable_sort():
    from sceneego_b200.network.voxel_net_depth import camera_frame_order
    rng = np.random.default_rng(0)
    for n, k in [(1, 1), (9, 2), (64, 5), (64, 16), (33, 16)]:
        ids = rng.integers(0, k, n)
        order = camera_frame_order(ids)
        assert order.dtype == np.int32
        assert order.tolist() == [i for _, i in sorted((int(c), i) for i, c in enumerate(ids))]
    assert camera_frame_order([1, 0, 1, 0, 1]).tolist() == [1, 3, 0, 2, 4]


def _fake(n):
    return C.c_void_p(n)          # never dereferenced: every call below is refused before a launch


def test_c_entries_refuse_bad_arguments():
    from sceneego_b200 import _lib
    lib = _lib.load_library()
    lay = _lib.vol_layout(64, 1, 2)
    cal = (_lib.Calib * 2)()
    P = _fake(1 << 20)

    def unproject(feat=P, grids=P, calibs=cal, k=2, cams=P, order=P):
        rc = lib.sceneego_unproject_cameras_f32(feat, grids, calibs, k, cams, order, 2, 64, 64, 32, 64, C.c_float(2.0),
                                                IMG_H, IMG_W, P, None, None, 0, None)
        return rc, lib.sceneego_last_error().decode()

    def voxelize(depth=P, rays=P, k=2, cams=P, order=P):
        rc = lib.sceneego_voxelize_depth_cameras_f64(depth, 2, IMG_H, IMG_W, IMG_H, IMG_W, C.c_float(float("inf")), rays, k,
                                                     cams, order, IMG_H, IMG_W, 64, C.c_double(2.0), P, None,
                                                     C.byref(lay), 32, None)
        return rc, lib.sceneego_last_error().decode()

    for rc, msg in (unproject(k=0), unproject(k=17), unproject(k=-1), voxelize(k=0), voxelize(k=17)):
        assert rc == -1 and "n_cameras must be in [1, 16]" in msg
    for rc, msg in (unproject(cams=None), voxelize(cams=None)):
        assert rc == -1 and "null frame_camera" in msg
    for rc, msg in (unproject(feat=None), unproject(grids=None, calibs=None), voxelize(depth=None), voxelize(rays=None)):
        assert rc == -1 and "null argument" in msg


# ---- GPU: the camera-per-frame gather against one launch per camera -----------------------------------------------------
def _calibs(files, k):
    from sceneego_b200.utils.fisheye.FishEyeCalibrated import FishEyeCameraCalibrated
    return [FishEyeCameraCalibrated(f).calib_struct(IMG_W, IMG_H) for f in files[:k]]


def _ids(pattern, B, K, seed):
    if pattern == "equal":
        return np.full(B, K - 1, np.int32)
    if pattern == "sorted":
        return np.sort(np.arange(B) % K).astype(np.int32)
    if pattern == "interleaved":
        return (np.arange(B) % K).astype(np.int32)
    return np.random.default_rng(seed).integers(0, K, B).astype(np.int32)


def _layout(kind, V, B):
    from sceneego_b200 import _lib
    if kind == "plain":
        return _lib.vol_layout(V, 1, B), 40
    if kind == "s2d":
        return _lib.vol_layout_s2d(V, B), 33 * 8
    return _lib.vol_layout_zwin(V, B), 40


def _sentinel_volume(lay, ch):
    from sceneego_b200 import _lib
    vol = _lib.alloc_volume(lay, ch, "cuda")
    vol.view(torch.int16).fill_(-1)
    return vol


def _nan(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device="cuda")


GATHER_CASES = [
    # K, B, V, ids, frame_order NULL
    (1, 1, 64, "equal", False),
    (2, 9, 48, "interleaved", False),
    (5, 33, 64, "random", False),
    (16, 64, 64, "random", False),
    (2, 64, 64, "sorted", False),
    (5, 9, 96, "sorted", True),
    (16, 33, 48, "interleaved", True),
    (2, 64, 64, "equal", True),
    (5, 1, 96, "random", False),
    (16, 9, 64, "sorted", False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True], ids=["table", "fused"])
@pytest.mark.parametrize("case", GATHER_CASES, ids=[f"K{c[0]}-B{c[1]}-V{c[2]}-{c[3]}{'-noorder' if c[4] else ''}"
                                                     for c in GATHER_CASES])
def test_unproject_cameras_equals_one_launch_per_camera(case, fused, calib_files):
    from sceneego_b200 import _lib
    from sceneego_b200.network.voxel_net_depth import camera_frame_order
    from tests.test_gpu_v2v_exact import check_untouched
    K, B, V, pattern, no_order = case
    calibs = _calibs(calib_files, K)
    grids = torch.stack([_lib.project_voxels(c, V, 2.0, (IMG_H, IMG_W), "cuda")[1] for c in calibs])
    ids = _ids(pattern, B, K, seed=B * 31 + K)
    order = None if no_order else torch.from_numpy(camera_frame_order(ids)).cuda()
    d_ids = torch.from_numpy(ids).cuda()
    g = torch.Generator().manual_seed(B + V + K)
    feat = torch.randn(B, 64, 64, 32, generator=g).cuda()
    where = f"unproject_cameras K{K} B{B} V{V} {pattern} fused={fused} order={'NULL' if no_order else 'sorted'}"

    def run(out_f32, vol, lay, extra):
        _lib.unproject_cameras(feat, None if fused else grids, calibs, d_ids, order, V, 2.0, IMG_H, IMG_W, out_f32, vol,
                               lay, extra_zero_planes=extra)

    def run_ref(out_f32, vol_of, extra):
        """one sceneego_unproject_f32 launch per camera on that camera's frames, scattered back"""
        for k in range(K):
            fk = np.nonzero(ids == k)[0]
            if fk.size == 0:
                continue
            sub = feat[torch.from_numpy(fk).cuda()].contiguous()
            o = None if out_f32 is None else torch.empty(fk.size, 32, V, V, V, device="cuda")
            vol, lay = vol_of(fk.size) if vol_of is not None else (None, None)
            _lib.unproject(sub, None if fused else grids[k].contiguous(), calibs[k] if fused else None, V, 2.0, IMG_H,
                           IMG_W, o, vol, lay, extra_zero_planes=extra)
            if o is not None:
                out_f32[torch.from_numpy(fk).cuda()] = o
            else:
                yield fk, _lib.unpack_volume(vol, lay, fk.size, 33)

    out = _nan(B + 1, 32, V, V, V)
    run(out[:B], None, None, 0)
    ref = torch.empty(B, 32, V, V, V, device="cuda")
    for _ in run_ref(ref, None, 0):
        pass
    torch.cuda.synchronize()
    assert torch.equal(out[:B], ref), where + " f32 NCDHW"
    assert bool(torch.isnan(out[B:]).all()), where + ": the spare frame was written"
    del out, ref
    for kind in ("plain", "s2d", "zwin"):
        lay, ch = _layout(kind, V, B + 1)
        vol = _sentinel_volume(lay, ch)
        run(None, vol, lay, 1)
        got = _lib.unpack_volume(vol, lay, B, 33)
        want = torch.empty_like(got)
        for fk, sub in run_ref(None, lambda n: (_sentinel_volume(*_layout(kind, V, n)), _layout(kind, V, n)[0]), 1):
            want[torch.from_numpy(fk).cuda()] = sub
        torch.cuda.synchronize()
        assert torch.equal(got, want), f"{where} {kind} layout"
        assert not bool(got[:, 32].any()), f"{where} {kind}: the occupancy plane was not cleared"
        check_untouched(vol, lay, B, f"{where} {kind} layout")


# ---- GPU: the camera-per-frame voxelisation against the NumPy oracle -------------------------------------------------------
def _oracle_occ(depth, ray, V):
    return np.stack([orc.voxelize_depth(d, ray, V, 2.0) for d in depth])


@pytest.fixture(scope="module")
def oracle_rays(calib_files):
    return [orc.ray_table(orc.load_calibration(f), IMG_W, IMG_H) for f in calib_files[:3]]


VOX_CASES = [
    # maps, V, ids
    ("room+uniform", 64, [2, 0, 1, 1, 0, 2]),
    ("room", 48, [1, 1, 0, 2, 2, 0, 1, 0, 2]),
    ("raw-demo", 64, [1, 2, 0]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("out", ["f32", "plain", "s2d", "zwin"])
@pytest.mark.parametrize("case", VOX_CASES, ids=[c[0] + f"-V{c[1]}" for c in VOX_CASES])
def test_voxelize_cameras_equals_the_oracle(case, out, calib_files, oracle_rays):
    """Zero-depth pixels (outside the image circle) and the padded columns land on the zero-depth voxel; the raw path
    resizes 512x640 demo maps and clamps at 10 m inside the kernel."""
    from sceneego_b200 import _lib
    from sceneego_b200.network.voxel_net_depth import camera_frame_order
    name, V, ids = case
    ids = np.array(ids, np.int32)
    B = ids.size
    calibs = _calibs(calib_files, 3)
    rays = torch.stack([_lib.ray_table(c, "cuda") for c in calibs])
    for k in range(3):        # the device table is the oracle's, row-major
        assert np.array_equal(rays[k].permute(1, 0, 2).reshape(-1, 3).cpu().numpy(), oracle_rays[k])
    pre, cm = None, float("inf")
    if name == "raw-demo":
        gv = util.golden("voxel.npz")
        raw = np.stack([gv[f"{n}_raw"] for n in ("img_001000", "img_001796", "img_002376")]).astype(np.float32)
        raw[1, 100:140, 200:260] = 25.0                                   # beyond the clamp
        depth = torch.from_numpy(raw)
        host = np.stack([orc.preprocess_depth(r) for r in raw])
        pre, cm = (IMG_H, IMG_W), 10.0
    else:
        room = [synth.synthetic_depth_room(1, oracle_rays[k], seed=60 + b)[0] for b, k in enumerate(ids)]
        depth = torch.stack(room)
        if name == "room+uniform":
            depth[1] = synth.synthetic_depth_uniform(1, seed=3)[0]
            depth[4, :, :300] = 0.0
        host = depth.numpy()
    want = np.zeros((B, V, V, V), np.float32)
    for b, k in enumerate(ids):
        want[b] = _oracle_occ(host[b:b + 1], oracle_rays[k], V)[0]
    d_ids = torch.from_numpy(ids).cuda()
    order = torch.from_numpy(camera_frame_order(ids)).cuda()
    where = f"voxelize_cameras {name} V{V} {out}"
    if out == "f32":
        occ = torch.zeros(B + 1, V, V, V, device="cuda")
        occ[B] = float("nan")
        _lib.voxelize_depth_cameras(depth.cuda(), pre, cm, rays, d_ids, order, IMG_H, IMG_W, V, 2.0, occ[:B], None, None)
        torch.cuda.synchronize()
        assert np.array_equal(occ[:B].cpu().numpy(), want), where
        assert bool(torch.isnan(occ[B]).all()), where + ": the spare frame was written"
        return
    lay, ch = _layout(out, V, B + 1)
    vol = _lib.alloc_volume(lay, ch, "cuda")
    _lib.voxelize_depth_cameras(depth.cuda(), pre, cm, rays, d_ids, order, IMG_H, IMG_W, V, 2.0, None, vol, lay,
                                channel=32)
    got = _lib.unpack_volume(vol, lay, B, 33)[:, 32].cpu().numpy()
    assert np.array_equal(got, want), where
    if out == "zwin":        # the whole z-window cell: entry e of (x,y,z) is occ[x][y][z-3+e]
        from tests.test_gpu_v2v_exact import decode
        cells = decode(vol, lay, B, 40)[:, 32:].cpu().numpy()           # (B, 8 entries, V, V, V)
        pad = np.pad(want, ((0, 0), (0, 0), (0, 0), (3, 4)))
        for e in range(8):
            assert np.array_equal(cells[:, e], pad[..., e:e + V]), f"{where} entry {e}"
    assert not bool(vol[:, B * lay.frame_pitch + lay.guard:].any()), where + ": the spare frame was written"


# ---- GPU: the module against one module per camera -----------------------------------------------------------------------
def _state(with_intersection):
    return synth.synthetic_state_dict(synth.stage_state_shapes(with_intersection=with_intersection), seed=0,
                                      mode="random_bn")


def _module(calib, with_intersection=False, **kw):
    from sceneego_b200.network.voxel_net_depth import VoxelNetwork_depth
    cfg = util.load_config(batch_size=4)
    cfg.dataset.camera_calibration_path = calib
    cfg.model.with_intersection = with_intersection
    torch.manual_seed(0)
    net = VoxelNetwork_depth(cfg, device="cuda", v2v_chunk=4, **kw).eval()
    full = net.state_dict()
    full.update(_state(with_intersection))
    net.load_state_dict(full, strict=True)
    net.keep_logits = True
    return net


@pytest.fixture(scope="module")
def nets(calib_files):
    """(multi-camera module with cameras 05_08, shifted, scaled; the three per-camera modules), for both configs."""
    out = {}
    for inter in (False, True):
        files = calib_files[:3]
        net = _module(files[0], inter)
        assert [net.add_camera(files[1]), net.add_camera(files[2])] == [1, 2]
        per_cam = [_module(f, inter) for f in files]
        for nk in per_cam:
            nk.load_state_dict(net.state_dict())
        out[inter] = (net, per_cam)
    return out


def _inputs(B, seed, oracle_rays):
    feat = synth.synthetic_features(B, seed=seed).cuda()
    depth = torch.cat([synth.synthetic_depth_room(1, oracle_rays[b % 3], seed=seed + b) for b in range(B)])
    return feat, depth


def _call(net, path, feat, depth, ids, images=None):
    kw = {} if ids is None else {"camera_ids": ids}
    if path == "scene":                                    # `depth` holds the scene grids
        return net.lift(feat, net.grid_coord_proj_batch, net.coord_volumes, scene_volumes=depth, **kw)
    d = depth.cuda()
    if path == "raw":
        d = d[:, ::2, ::2].contiguous() * 3.0                  # 512 x 640 maps, some beyond the 10 m clamp
    if images is not None:
        return net(images, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=d, **kw)
    return net.lift(feat, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=d, **kw)


def _set(nets_list, **attrs):
    for n in nets_list:
        for k, v in attrs.items():
            setattr(n, k, v)


def _check_spec(net, per_cam, path, feat, depth, ids, where, images=None):
    if path == "scene":
        # one set of scene grids for every module: on this path only the gather depends on the camera
        from sceneego_b200 import _lib
        occ = torch.zeros(feat.shape[0], 64, 64, 64, device="cuda")
        _lib.voxelize_depth(depth.cuda().contiguous(), net._ray_dev, IMG_H, IMG_W, 64, 2.0, occ, None, None)
        depth = occ
    got = _call(net, path, feat, depth, ids, images)
    got_logits = net.last_logits
    for k, nk in enumerate(per_cam):
        ref = _call(nk, path, feat, depth, None, images)
        fk = torch.from_numpy(np.nonzero(np.asarray(ids) == k)[0]).cuda()
        if fk.numel() == 0:
            continue
        for name, a, b in (("keypoints", got[0], ref[0]), ("output #2", got[1], ref[1]), ("output #3", got[2], ref[2]),
                           ("logits", got_logits, nk.last_logits)):
            assert torch.equal(a[fk], b[fk]), f"{where}: {name} of camera {k}'s frames"
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True], ids=["table", "fused"])
@pytest.mark.parametrize("path", ["depth", "raw", "scene"])
def test_lift_with_camera_ids_equals_per_camera_modules(nets, oracle_rays, path, fused):
    net, per_cam = nets[False]
    everyone = [net] + per_cam
    _set(everyone, fused_projection=fused, depth_preprocess=(IMG_H, IMG_W, 10.0) if path == "raw" else None)
    try:
        feat, depth = _inputs(6, 70, oracle_rays)           # two V2V chunks of 4 and 2 frames
        with torch.no_grad():
            for ids in ([2, 0, 1, 1, 0, 2], np.array([1, 1, 1, 2, 2, 0]), torch.tensor([0, 2, 2, 2, 0, 0])):
                _check_spec(net, per_cam, path, feat, depth, ids, f"lift {path} fused={fused} ids={list(ids)}")
    finally:
        _set(everyone, fused_projection=False, depth_preprocess=None)


@pytest.mark.gpu
def test_camera_ids_with_intersection(nets, oracle_rays):
    net, per_cam = nets[True]
    feat, depth = _inputs(5, 80, oracle_rays)
    with torch.no_grad():
        _check_spec(net, per_cam, "depth", feat, depth, [1, 0, 2, 2, 1], "with_intersection")


@pytest.mark.gpu
@pytest.mark.parametrize("handoff", [False, True])
def test_forward_with_camera_ids(nets, oracle_rays, handoff):
    net, per_cam = nets[False]
    _set([net] + per_cam, backbone_handoff=handoff)
    try:
        g = torch.Generator().manual_seed(5)
        images = torch.randn(3, 3, 256, 256, generator=g).cuda()
        feat, depth = _inputs(3, 90, oracle_rays)
        with torch.no_grad():
            _check_spec(net, per_cam, "depth", feat, depth, [2, 1, 0], f"forward handoff={handoff}", images=images)
    finally:
        _set([net] + per_cam, backbone_handoff=False)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True], ids=["table", "fused"])
def test_camera_ids_all_zero_equal_none(nets, oracle_rays, fused):
    net, _ = nets[False]
    net.fused_projection = fused
    try:
        feat, depth = _inputs(6, 100, oracle_rays)
        with torch.no_grad():
            a = net.lift(feat, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=depth.cuda())
            la = net.last_logits
            b = net.lift(feat, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=depth.cuda(),
                         camera_ids=[0] * 6)
        for x, y in zip(a[:3] + (la,), b[:3] + (net.last_logits,)):
            assert torch.equal(x, y)
    finally:
        net.fused_projection = False


@pytest.mark.gpu
def test_module_refuses_bad_camera_arguments(nets, oracle_rays, calib_files):
    from sceneego_b200 import _lib
    net, _ = nets[False]
    feat, depth = _inputs(3, 110, oracle_rays)
    d = depth.cuda()
    with pytest.raises(_lib.SceneEgoError, match="host-side sequence"):
        net.lift(feat, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=d,
                 camera_ids=torch.tensor([0, 1, 2], device="cuda"))
    with pytest.raises(_lib.SceneEgoError, match=r"lie in \[0, 3\)"):
        net.lift(feat, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=d, camera_ids=[0, 3, 1])
    foreign = net.grid_coord_proj_batch.clone()
    with pytest.raises(_lib.SceneEgoError, match="per-camera tables come from add_camera"):
        net.lift(feat, foreign, net.coord_volumes, depth_map_batch=d, camera_ids=[0, 1, 2])
    # the reference attributes stay camera 0's
    assert net.fisheye_camera_model is net.cameras[0] and len(net.cameras) == 3
    own = _module(calib_files[0])
    assert torch.equal(net.grid_coord_proj_batch, own.grid_coord_proj_batch) and np.array_equal(net.ray, own.ray)


@pytest.mark.gpu
def test_add_camera_limits_and_odd_volume_size(calib_files, tmp_path):
    from sceneego_b200 import _lib
    from sceneego_b200.network.voxel_net_depth import VoxelNetwork_depth
    from sceneego_b200.utils.fisheye.FishEyeCalibrated import FishEyeCameraCalibrated
    net = VoxelNetwork_depth(util.load_config(batch_size=1, volume_size=32), device="cuda", v2v_chunk=1).eval()
    with pytest.raises(_lib.SceneEgoError, match="differs from the module's"):
        VoxelNetwork_depth.add_camera(net, _write_calib(tmp_path / "small.json", size=(640, 512)))
    assert net.add_camera(FishEyeCameraCalibrated(calib_files[1])) == 1
    for f in calib_files[2:]:
        net.add_camera(f)
    assert len(net.cameras) == 16 and tuple(net._cam_grids.shape) == (16, 32 ** 3, 2)
    assert tuple(net._cam_rays.shape) == (16, IMG_H, IMG_W, 3)
    with pytest.raises(_lib.SceneEgoError, match="at most 16 cameras"):
        net.add_camera(calib_files[1])
    # an odd volume size puts a voxel centre on the optical axis: the same error as the constructor's
    odd = net
    odd.cameras, odd._cam_calibs = odd.cameras[:1], odd._cam_calibs[:1]
    odd._cam_grids = odd._cam_rays = None
    odd.volume_size = 31
    odd.coord_volume = odd.build_coord_volume()
    with pytest.raises(Exception, match="norm is zero!"):
        odd.add_camera(calib_files[1])


@pytest.mark.gpu
def test_graph_replays_with_a_new_assignment(calib_files, oracle_rays):
    """graph_max_batch: the ids live in a static buffer refilled before each replay; a new assignment does not capture
    again, and the frames come out as the per-camera modules' eager ones."""
    files = calib_files[:3]
    net = _module(files[0], graph_max_batch=4)
    net.add_camera(files[1])
    net.add_camera(files[2])
    per_cam = [_module(f) for f in files]
    feat, depth = _inputs(4, 120, oracle_rays)
    with torch.no_grad():
        for i, ids in enumerate(([0, 1, 2, 0], [2, 2, 1, 0], [1, 0, 1, 0])):
            _check_spec(net, per_cam, "depth", feat, depth, ids, f"graph replay {ids}")
            assert len(net._graphs) == 1, "a new camera assignment captured again"
        _check_spec(net, per_cam, "depth", feat, depth, [0, 0, 0, 0], "graph all zero")
        assert len(net._graphs) == 1
        net.lift(feat, net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=depth.cuda())
        assert len(net._graphs) == 2                       # camera mode off is its own capture
        net.add_camera(files[1])                           # new stacked tables: a new capture
        _check_spec(net, per_cam + [per_cam[1]], "depth", feat, depth, [3, 0, 2, 1], "graph after add_camera")
        assert len(net._graphs) == 3


@pytest.mark.gpu
def test_host_pipeline_with_camera_ids(nets, oracle_rays):
    from sceneego_b200.pipeline import HostStagePipeline
    net, _ = nets[False]
    B = 8
    feats = [synth.synthetic_features(B, seed=130 + i).pin_memory() for i in range(2)]
    depths = [_inputs(B, 140 + i, oracle_rays)[1].pin_memory() for i in range(2)]
    ids = [np.array([2, 0, 1, 1, 0, 2, 2, 1]), [0, 1, 2, 0, 1, 2, 0, 1]]
    with torch.no_grad():
        for ramp in (64, 8):                                # plain, then the first batch ramped in parts 2, 2, 4
            pipe = HostStagePipeline(net)
            pipe.ramp_min_batch = ramp
            outs = [o.clone() for o in pipe.run(list(zip(feats, depths, ids)))]
            for i in range(2):
                parts = [(0, 2), (2, 4), (4, 8)] if (ramp == 8 and i == 0) else [(0, B)]
                ref = torch.cat([net.lift(feats[i][s0:s1].cuda(), net.grid_coord_proj_batch, net.coord_volumes,
                                          depth_map_batch=depths[i][s0:s1].cuda(),
                                          camera_ids=ids[i][s0:s1])[0] for s0, s1 in parts]).cpu()
                assert torch.equal(outs[i], ref), (ramp, i)


@pytest.mark.gpu
def test_camera_ids_parity_with_the_oracle(nets, calib_files):
    """End to end against the CPU oracle run with each camera's StageTables: the 0.5 mm MPJPE gate."""
    net, _ = nets[False]
    tables = [orc.StageTables(f, 64, 2.0) for f in calib_files[:3]]
    ids = [1, 2, 0]
    feat = synth.synthetic_features(3, seed=150)
    depth = torch.cat([synth.synthetic_depth_room(1, tables[k].ray, seed=151 + b) for b, k in enumerate(ids)])
    with torch.no_grad():
        kp = net.lift(feat.cuda(), net.grid_coord_proj_batch, net.coord_volumes, depth_map_batch=depth.cuda(),
                      camera_ids=ids)[0].cpu().numpy()
    sd = _state(False)
    for b, k in enumerate(ids):
        ref = orc.stage_forward(tables[k], sd, feat[b:b + 1], depth_batch=depth[b:b + 1])[0].numpy()
        err = orc.mpjpe(kp[b:b + 1], ref) * 1000.0
        print(f"camera {k}: MPJPE vs oracle {err:.4f} mm")
        assert err <= 0.5, (k, err)


# ---- both storage builds -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.skipif(F16_RUN, reason="already running on the fp16-storage build")
def test_cameras_with_fp16_storage_build():
    """This file's GPU tests on libsceneego_b200_f16.so (one activation dtype per process: a subprocess)."""
    env = dict(os.environ, SCENEEGO_ACT_DTYPE="f16", PYTHONPATH=util.ROOT)
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_cameras.py", "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider"], cwd=util.ROOT, env=env, capture_output=True, text=True, timeout=3000)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert " passed" in tail.splitlines()[-1]

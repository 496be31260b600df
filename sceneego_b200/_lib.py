"""ctypes binding of libsceneego_b200.so (the C-ABI of include/sceneego_b200.h).

There is NO fallback: if the CUDA library cannot be loaded, or a tensor is not
on a CUDA device, every op raises.  PyTorch is used only for device memory and
streams; all compute goes through the extern "C" entry points.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# Storage type of V2V activations / packed weights: "bf16" (default; BASELINE configs[1]) or "f16" (the same sources
# compiled with -DSCENEEGO_ACT_F16: 3 more mantissa bits, saturating stores).  One per process, chosen by the
# environment variable SCENEEGO_ACT_DTYPE or set_act_dtype() before the library is first loaded.
_ACT = os.environ.get("SCENEEGO_ACT_DTYPE", "bf16").lower()
LIB_PATHS = {"bf16": os.path.join(_HERE, "libsceneego_b200.so"), "f16": os.path.join(_HERE, "libsceneego_b200_f16.so")}
LIB_PATH = LIB_PATHS["bf16"]


def set_act_dtype(name: str) -> None:
    global _ACT
    name = {"fp16": "f16", "float16": "f16", "bfloat16": "bf16"}.get(name.lower(), name.lower())
    if name not in LIB_PATHS:
        raise SceneEgoError(f"unknown activation dtype {name!r} (bf16 or f16)")
    if _lib is not None and name != _ACT:
        raise SceneEgoError("the activation dtype is fixed once the library is loaded (one per process)")
    _ACT = name


def act_dtype_name() -> str:
    return _ACT


def act_torch_dtype():
    return torch.float16 if _ACT == "f16" else torch.bfloat16

SYMBOLS = [
    "sceneego_abi_version", "sceneego_act_dtype", "sceneego_last_error", "sceneego_ray_table_f64", "sceneego_project_voxels_f32",
    "sceneego_feature_conv1x1_f32", "sceneego_features_upsample_pad_f32", "sceneego_vol_layout_make",
    "sceneego_unproject_f32", "sceneego_voxelize_depth_f64", "sceneego_pack_volume_bf16",
    "sceneego_unpack_volume_f32", "sceneego_v2v_pack_conv", "sceneego_v2v_run", "sceneego_v2v_run_profile",
    "sceneego_v2v_last_launch_count", "sceneego_softargmax_workspace_bytes", "sceneego_softargmax3d_f32",
    "sceneego_world2camera_f32", "sceneego_grid_sample_f32", "sceneego_vol_layout_make_s2d",
    "sceneego_v2v_stem_s2d_weight_bytes", "sceneego_v2v_pack_stem_s2d", "sceneego_v2v_pack_conv_march", "sceneego_voxelize_depth_raw_f64", "sceneego_intersect_bf16", "sceneego_pose_errors_f64",
    "sceneego_voxelize_depth_dataset_f64", "sceneego_vol_layout_make_zwin", "sceneego_occ_expand_zwin_bf16", "sceneego_v2v_stem_march_weight_bytes",
    "sceneego_v2v_pack_stem_march", "sceneego_handoff_weight_bytes", "sceneego_handoff_workspace_bytes", "sceneego_handoff_pack",
    "sceneego_backbone_handoff_f32", "sceneego_voxelize_points", "sceneego_voxelize_scan",
]


class Calib(C.Structure):
    _fields_ = [("cx", C.c_double), ("cy", C.c_double), ("c2w", C.c_double * 7), ("w2c", C.c_double * 11),
                ("width", C.c_int32), ("height", C.c_int32)]


class VolLayout(C.Structure):
    _fields_ = [("side", C.c_int32), ("pad", C.c_int32), ("pitch_y", C.c_int32), ("pitch_x", C.c_int32),
                ("guard", C.c_int32), ("frame_pitch", C.c_int32), ("plane_stride", C.c_int64),
                ("s2d", C.c_int32), ("zwin", C.c_int32)]


class V2VOp(C.Structure):
    _fields_ = [("type", C.c_int32), ("flags", C.c_int32), ("ksize", C.c_int32), ("cin", C.c_int32),
                ("cout", C.c_int32), ("cout_real", C.c_int32), ("src", C.c_int32), ("dst", C.c_int32),
                ("res", C.c_int32), ("impl", C.c_int32), ("xstack", C.c_int32), ("cta_pair", C.c_int32), ("w_offset", C.c_int64),
                ("b_offset", C.c_int64), ("src2", C.c_int32), ("cin2", C.c_int32),
                ("lay_src", VolLayout), ("lay_dst", VolLayout)]


OP_CONV, OP_MAXPOOL2, OP_DECONV2, OP_STEM7_S2D, OP_TAIL_MLP, OP_CONV3_MARCH, OP_STEM7_MARCH = 0, 1, 2, 3, 4, 5, 6
F_RELU, F_RESIDUAL, F_ADD_AFTER, F_OUT_F32 = 1, 2, 4, 8

_lib = None


class SceneEgoError(RuntimeError):
    pass


def load_library(path: Optional[str] = None) -> C.CDLL:
    """Load the shared library (no compute is performed)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATHS[_ACT]
    if not os.path.exists(p):
        raise SceneEgoError(
            f"{p} not found: build it with `python -m sceneego_b200.build` "
            "(sceneego_b200 has no CPU or PyTorch fallback)")
    lib = C.CDLL(p)
    lib.sceneego_last_error.restype = C.c_char_p
    lib.sceneego_vol_layout_make.restype = C.c_int64
    lib.sceneego_vol_layout_make_s2d.restype = C.c_int64
    lib.sceneego_vol_layout_make_zwin.restype = C.c_int64
    lib.sceneego_v2v_stem_march_weight_bytes.restype = C.c_size_t
    lib.sceneego_handoff_weight_bytes.restype = C.c_size_t
    lib.sceneego_handoff_workspace_bytes.restype = C.c_size_t
    lib.sceneego_v2v_stem_s2d_weight_bytes.restype = C.c_size_t
    lib.sceneego_softargmax_workspace_bytes.restype = C.c_size_t
    if lib.sceneego_abi_version() != 5:
        raise SceneEgoError("libsceneego_b200.so ABI version mismatch")
    if path is None and lib.sceneego_act_dtype() != (1 if _ACT == "f16" else 0):
        raise SceneEgoError(f"{p} was not compiled for {_ACT} activations")
    if path is None:
        _lib = lib
    return lib


def _check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load_library().sceneego_last_error().decode()
        if rc == -3:
            raise Exception("norm is zero!")  # same exception text as FishEyeCalibrated.py:177
        raise SceneEgoError(f"{what} failed (code {rc}): {msg}")


def _ptr(t: Optional[torch.Tensor], device: Optional[torch.device] = None) -> C.c_void_p:
    if t is None:
        return C.c_void_p(0)
    if not t.is_cuda:
        raise SceneEgoError("sceneego_b200 ops need CUDA tensors (no CPU fallback)")
    if device is not None and t.device != device:
        raise SceneEgoError(f"sceneego_b200 op: tensors on different devices ({t.device} vs {device})")
    if not t.is_contiguous():
        raise SceneEgoError("sceneego_b200 ops need contiguous tensors")
    return C.c_void_p(t.data_ptr())


def _as_device(device) -> torch.device:
    d = torch.device(device)
    if d.type != "cuda":
        raise SceneEgoError("sceneego_b200 ops need a CUDA device (no CPU fallback)")
    return d if d.index is not None else torch.device("cuda", torch.cuda.current_device())


class on_device:
    """Make `device` the current CUDA device for the duration of a C-ABI call.  The library never calls
    cudaSetDevice: kernels launch on the calling thread's current device, so the binding selects the device the
    tensors live on (a module built with device='cuda:1' works without torch.cuda.set_device(1))."""

    def __init__(self, device):
        self.device = _as_device(device)
        self.prev = None

    def __enter__(self):
        cur = torch.cuda.current_device()
        if cur != self.device.index:
            self.prev = cur
            torch.cuda.set_device(self.device.index)
        return self.device

    def __exit__(self, *exc):
        if self.prev is not None:
            torch.cuda.set_device(self.prev)
        return False


def _stream(device=None) -> C.c_void_p:
    """torch's current stream ON THE GIVEN DEVICE (a tensor or a device; default: the current device)."""
    if isinstance(device, torch.Tensor):
        device = device.device
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _call(name: str, anchor, *args) -> None:
    """lib.<name>(*args, stream): `anchor` (tensor or device) fixes the device and the stream; tensor arguments become
    raw pointers after a same-device / contiguity check, None becomes NULL."""
    dev = _as_device(anchor.device if isinstance(anchor, torch.Tensor) else anchor)
    conv = [_ptr(a, dev) if isinstance(a, torch.Tensor) else a for a in args]
    with on_device(dev):
        rc = getattr(load_library(), name)(*conv, _stream(dev))
    _check(rc, name.replace("sceneego_", ""))


def make_calib(cx, cy, c2w, w2c, width, height) -> Calib:
    c = Calib()
    c.cx, c.cy = float(cx), float(cy)
    for i in range(7):
        c.c2w[i] = float(c2w[i])
    for i in range(11):
        c.w2c[i] = float(w2c[i])
    c.width, c.height = int(width), int(height)
    return c


def vol_layout(side: int, pad: int, batch: int) -> VolLayout:
    lay = VolLayout()
    rc = load_library().sceneego_vol_layout_make(int(side), int(pad), int(batch), C.byref(lay))
    if rc < 0:
        raise SceneEgoError("vol_layout_make: bad arguments")
    return lay


def vol_layout_s2d(full_side: int, batch: int) -> VolLayout:
    """Space-to-depth layout of the stem input (8 parity sub-volumes of side full_side/2, pad 2)."""
    lay = VolLayout()
    rc = load_library().sceneego_vol_layout_make_s2d(int(full_side), int(batch), C.byref(lay))
    if rc < 0:
        raise SceneEgoError("vol_layout_make_s2d: bad arguments")
    return lay


def vol_layout_zwin(side: int, batch: int) -> VolLayout:
    """Input layout of the marching stem: plain planar, pad 3, plane 4 = z-window occupancy (lay.zwin = 1)."""
    lay = VolLayout()
    rc = load_library().sceneego_vol_layout_make_zwin(int(side), int(batch), C.byref(lay))
    if rc < 0:
        raise SceneEgoError("vol_layout_make_zwin: bad arguments")
    return lay


def alloc_volume(lay: VolLayout, channels: int, device) -> torch.Tensor:
    """Zero-initialised planar padded volume of the 16-bit activation type: (C/8, plane_stride, 8)."""
    assert channels % 8 == 0
    return torch.zeros(channels // 8, lay.plane_stride, 8, dtype=act_torch_dtype(), device=device)


# ---- thin per-op wrappers (argument checking lives in C) ---------------------
def ray_table(calib: Calib, device) -> torch.Tensor:
    device = _as_device(device)
    out = torch.empty(calib.height, calib.width, 3, dtype=torch.float64, device=device)
    _call("sceneego_ray_table_f64", out, C.byref(calib), out)
    return out


def project_voxels(calib: Calib, volume_size: int, cuboid_side: float, heatmap_shape, device):
    device = _as_device(device)
    n = volume_size ** 3
    px = torch.empty(n, 2, dtype=torch.float32, device=device)
    grid = torch.empty(n, 2, dtype=torch.float32, device=device)
    status = torch.zeros(1, dtype=torch.int32, device=device)
    _call("sceneego_project_voxels_f32", px, C.byref(calib), int(volume_size), C.c_float(cuboid_side),
          int(heatmap_shape[0]), int(heatmap_shape[1]), px, grid, status)
    if int(status.item()) != 0:
        raise Exception("norm is zero!")
    return px, grid


def world2camera(calib: Calib, points: torch.Tensor) -> torch.Tensor:
    n = points.shape[0]
    px = torch.empty(n, 2, dtype=torch.float32, device=points.device)
    status = torch.zeros(1, dtype=torch.int32, device=points.device)
    _call("sceneego_world2camera_f32", points, C.byref(calib), points, n, px, status)
    if int(status.item()) != 0:
        raise Exception("norm is zero!")
    return px


def grid_sample(img: torch.Tensor, grid: torch.Tensor, grid_batch_stride: int) -> torch.Tensor:
    b, c, h, w = img.shape
    n = grid.shape[-3] if grid.dim() == 4 else grid.shape[0]
    if grid.device != img.device:
        raise SceneEgoError("grid_sample: image and grid on different devices")
    out = torch.empty(b, c, n, dtype=torch.float32, device=img.device)
    _call("sceneego_grid_sample_f32", img, img, C.c_void_p(grid.data_ptr()), C.c_int64(grid_batch_stride), b, c, h, w,
          n, out)
    return out


def feature_conv1x1(feat: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    b, cin, h, w = feat.shape
    cout = weight.shape[0]
    if out is None:
        out = torch.empty(b, h, w, cout, dtype=torch.float32, device=feat.device)
    elif tuple(out.shape) != (b, h, w, cout) or out.dtype != torch.float32:
        raise SceneEgoError("feature_conv1x1: bad output buffer")
    _call("sceneego_feature_conv1x1_f32", feat, feat, weight.reshape(cout, cin), bias, out, b, cin, cout, h, w)
    return out


def features_upsample_pad(feat_cl: torch.Tensor, up: int, pad: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    b, h, w, c = feat_cl.shape
    if out is None:
        out = torch.empty(b, c, up, up + 2 * pad, dtype=torch.float32, device=feat_cl.device)
    elif tuple(out.shape) != (b, c, up, up + 2 * pad) or out.dtype != torch.float32 or not out.is_contiguous():
        raise SceneEgoError("features_upsample_pad: bad output buffer")
    _call("sceneego_features_upsample_pad_f32", feat_cl, feat_cl, out, b, c, h, w, up, pad)
    return out


def unproject(feat_cl: torch.Tensor, grid: Optional[torch.Tensor], calib: Optional[Calib], volume_size: int,
              cuboid_side: float, img_h: int, img_w: int, out_f32: Optional[torch.Tensor],
              out_bf16: Optional[torch.Tensor], lay: Optional[VolLayout], extra_zero_planes: int = 0) -> None:
    b, h, w, c = feat_cl.shape
    _call("sceneego_unproject_f32", feat_cl, feat_cl, grid, C.byref(calib) if calib is not None else None, b, h, w, c,
          int(volume_size), C.c_float(cuboid_side), int(img_h), int(img_w), out_f32, out_bf16,
          C.byref(lay) if lay is not None else None, int(extra_zero_planes))


def voxelize_depth(depth: torch.Tensor, ray: torch.Tensor, img_h: int, img_w: int, volume_size: int,
                   cuboid_side: float, occ_f32: Optional[torch.Tensor], occ_bf16: Optional[torch.Tensor],
                   lay: Optional[VolLayout], channel: int = 0) -> None:
    b, h, w = depth.shape
    _call("sceneego_voxelize_depth_f64", depth, depth, b, h, w, ray, int(img_h), int(img_w), int(volume_size),
          C.c_double(cuboid_side), occ_f32, occ_bf16, C.byref(lay) if lay is not None else None, int(channel))


def voxelize_depth_raw(depth_raw: torch.Tensor, pre_hw, clamp_max: float, ray: torch.Tensor, img_h: int, img_w: int,
                       volume_size: int, cuboid_side: float, occ_f32: Optional[torch.Tensor],
                       occ_bf16: Optional[torch.Tensor], lay: Optional[VolLayout], channel: int = 0) -> None:
    """Raw depth maps: the dataset's nearest resize to `pre_hw` and clamp fused into the NETWORK's voxelisation."""
    b, h, w = depth_raw.shape
    _call("sceneego_voxelize_depth_raw_f64", depth_raw, depth_raw, b, h, w, int(pre_hw[0]), int(pre_hw[1]),
          C.c_float(clamp_max), ray, int(img_h), int(img_w), int(volume_size), C.c_double(cuboid_side), occ_f32,
          occ_bf16, C.byref(lay) if lay is not None else None, int(channel))


def voxelize_depth_dataset(depth_raw: torch.Tensor, pre_hw, clamp_max: float, ray: torch.Tensor, volume_size: int,
                           cuboid_side: float, occ_f32: torch.Tensor) -> None:
    """The DATASET's voxelisation (dataset/real_depth_utils.py:29-60): map times ray table pixel for pixel, no squash
    to H x H and no padded columns; the dataset's resize to `pre_hw` and clamp fused into the load."""
    b, h, w = depth_raw.shape
    if tuple(ray.shape) != (int(pre_hw[0]), int(pre_hw[1]), 3):
        raise SceneEgoError("voxelize_depth_dataset: the ray table must be (pre_h, pre_w, 3)")
    _call("sceneego_voxelize_depth_dataset_f64", depth_raw, depth_raw, b, h, w, int(pre_hw[0]), int(pre_hw[1]),
          C.c_float(clamp_max), ray, int(volume_size), C.c_double(cuboid_side), occ_f32)


def voxelize_points(points: torch.Tensor, offsets: torch.Tensor, volume_size: int, cuboid_side: float,
                    occ_f32: torch.Tensor) -> None:
    """Ragged batch of camera-space clouds -> occupancy (point_cloud_to_voxel_numpy, network/voxel_net_depth.py:207-222):
    points (N,3) float64 or float32 CUDA (computed in that precision), offsets (B+1,) int64 (frame b owns points
    [offsets[b], offsets[b+1]); a CPU tensor is checked on the host and copied, a CUDA one is copied to the host to be
    checked), occ_f32 (B,V,V,V) f32 zero-initialised; occupied voxels are set to 1."""
    if not isinstance(points, torch.Tensor) or points.dtype not in (torch.float64, torch.float32):
        raise SceneEgoError(f"voxelize_points: points must be a float64 or float32 tensor, got "
                            f"{getattr(points, 'dtype', type(points).__name__)}")
    if points.dim() != 2 or points.shape[1] != 3:
        raise SceneEgoError(f"voxelize_points: points must have shape (N, 3), got {tuple(points.shape)}")
    if not isinstance(offsets, torch.Tensor) or offsets.dtype != torch.int64 or offsets.dim() != 1 or offsets.numel() < 1:
        raise SceneEgoError("voxelize_points: offsets must be a 1-D int64 tensor of B + 1 entries")
    if not points.is_cuda:
        raise SceneEgoError("voxelize_points: points must be a CUDA tensor (no CPU fallback)")
    b, v = offsets.numel() - 1, int(volume_size)
    if (not isinstance(occ_f32, torch.Tensor) or occ_f32.dtype != torch.float32 or tuple(occ_f32.shape) != (b, v, v, v)
            or not occ_f32.is_cuda or occ_f32.device != points.device):
        raise SceneEgoError(f"voxelize_points: occ_f32 must be a float32 ({b}, {v}, {v}, {v}) tensor on {points.device}")
    o = offsets.cpu()
    n = points.shape[0]
    if int(o[0]) < 0 or int(o[-1]) > n or bool((o[1:] < o[:-1]).any()):
        raise SceneEgoError(f"voxelize_points: offsets must be non-decreasing within [0, {n}]")
    if b == 0 or int(o[-1]) == int(o[0]):
        return                                       # nothing to scatter (an empty tensor may have no storage)
    d_off = offsets if offsets.is_cuda and offsets.device == points.device else o.to(points.device)
    _call("sceneego_voxelize_points", points, points, int(points.dtype == torch.float64), d_off.contiguous(), b, v,
          C.c_double(cuboid_side), occ_f32)


def voxelize_scan(scan: torch.Tensor, cam_from_world: torch.Tensor, volume_size: int, cuboid_side: float,
                  occ_f32: torch.Tensor) -> None:
    """One world-space scan seen from B camera poses -> B occupancy grids in one launch, without a transformed copy of
    the scan: scan (N,3) float64 or float32 CUDA (computed in that precision), cam_from_world (B,4,4) of the scan's
    dtype, CPU or CUDA (checked on the host: finite, bottom row exactly (0,0,0,1); the upper (3,4) block is applied as
    given), occ_f32 (B,V,V,V) f32 zero-initialised; occupied voxels are set to 1."""
    if not isinstance(scan, torch.Tensor) or scan.dtype not in (torch.float64, torch.float32):
        raise SceneEgoError(f"voxelize_scan: scan must be a float64 or float32 tensor, got "
                            f"{getattr(scan, 'dtype', type(scan).__name__)}")
    if scan.dim() != 2 or scan.shape[1] != 3:
        raise SceneEgoError(f"voxelize_scan: scan must have shape (N, 3), got {tuple(scan.shape)}")
    if not isinstance(cam_from_world, torch.Tensor) or cam_from_world.dim() != 3 or tuple(cam_from_world.shape[1:]) != (4, 4):
        raise SceneEgoError(f"voxelize_scan: cam_from_world must be a (B, 4, 4) tensor, got "
                            f"{tuple(getattr(cam_from_world, 'shape', ())) or type(cam_from_world).__name__}")
    if cam_from_world.dtype != scan.dtype:
        raise SceneEgoError(f"voxelize_scan: cam_from_world must have the scan's dtype {scan.dtype}, got "
                            f"{cam_from_world.dtype} (the transform runs in the scan's precision; cast explicitly)")
    pose = cam_from_world.detach().cpu()
    if not bool(torch.isfinite(pose).all()):
        raise SceneEgoError("voxelize_scan: cam_from_world has non-finite entries")
    bottom = torch.tensor([0.0, 0.0, 0.0, 1.0], dtype=pose.dtype)
    if not bool((pose[:, 3, :] == bottom).all()):
        raise SceneEgoError("voxelize_scan: the bottom row of every cam_from_world must be exactly (0, 0, 0, 1)")
    b, v = pose.shape[0], int(volume_size)
    if (not isinstance(occ_f32, torch.Tensor) or occ_f32.dtype != torch.float32
            or tuple(occ_f32.shape) != (b, v, v, v)):
        raise SceneEgoError(f"voxelize_scan: occ_f32 must be a float32 ({b}, {v}, {v}, {v}) tensor")
    if not scan.is_cuda:
        raise SceneEgoError("voxelize_scan: scan must be a CUDA tensor (no CPU fallback)")
    if not occ_f32.is_cuda or occ_f32.device != scan.device:
        raise SceneEgoError(f"voxelize_scan: occ_f32 must be on {scan.device}")
    if b == 0 or scan.shape[0] == 0:
        return                                       # nothing to scatter (an empty tensor may have no storage)
    d_pose = pose[:, :3, :].contiguous().to(scan.device)
    _call("sceneego_voxelize_scan", scan, scan, int(scan.dtype == torch.float64), C.c_int64(scan.shape[0]), d_pose, b, v,
          C.c_double(cuboid_side), occ_f32)


def occ_expand_zwin(occ_f32: torch.Tensor, vol: torch.Tensor, lay: VolLayout, channel: int) -> None:
    """Plain (B,V,V,V) f32 occupancy grid -> the z-window occupancy plane of `channel` in the marching stem's input
    (every real cell written); the grid is left all-zero for the next batch."""
    b = occ_f32.shape[0]
    if occ_f32.dtype != torch.float32 or not occ_f32.is_contiguous() or tuple(occ_f32.shape[1:]) != (lay.side,) * 3:
        raise SceneEgoError("occ_expand_zwin: needs a contiguous (B,V,V,V) f32 grid")
    _call("sceneego_occ_expand_zwin_bf16", occ_f32, occ_f32, vol, C.byref(lay), int(b), int(channel))


def intersect(vol_bf16: torch.Tensor, lay: VolLayout, batch: int, channels: int) -> None:
    """channels [c,2c) = channels [0,c) * occupancy (channel 2c), in place (with_intersection)."""
    _call("sceneego_intersect_bf16", vol_bf16, vol_bf16, C.byref(lay), int(batch), int(channels))


def pose_errors(pred: torch.Tensor, gt: torch.Tensor, scale: bool = True, want_aligned: bool = False):
    """Per-frame MPJPE and PA-MPJPE (fp64) of pred (B,J,3) f32 or f64 (dtype kept, like the reference's NumPy)
    against gt (B,J,3) f64; optionally the aligned poses, the ground truth align_skeleton returns and the
    (c, R, t) transforms."""
    b, j = pred.shape[0], pred.shape[1]
    pred = pred.contiguous()
    if pred.dtype != torch.float64:
        pred = pred.float()
    gt = gt.contiguous().double()
    mp = torch.empty(b, dtype=torch.float64, device=pred.device)
    pa = torch.empty(b, dtype=torch.float64, device=pred.device)
    al = torch.empty(b, j, 3, dtype=torch.float64, device=pred.device) if want_aligned else None
    go = torch.empty(b, j, 3, dtype=torch.float64, device=pred.device) if want_aligned else None
    tr = torch.empty(b, 13, dtype=torch.float64, device=pred.device) if want_aligned else None
    _call("sceneego_pose_errors_f64", pred, pred, int(pred.dtype == torch.float64), gt, b, j, int(bool(scale)), mp, pa,
          al, go, tr)
    return mp, pa, al, go, tr


def pack_volume(x: torch.Tensor, out_bf16: torch.Tensor, lay: VolLayout, c_offset: int = 0) -> None:
    b, c = x.shape[:2]
    _call("sceneego_pack_volume_bf16", x, x, b, c, int(c_offset), out_bf16, C.byref(lay))


def unpack_volume(vol_bf16: torch.Tensor, lay: VolLayout, batch: int, channels: int) -> torch.Tensor:
    s = 2 * lay.side if lay.s2d else lay.side
    out = torch.empty(batch, channels, s, s, s, dtype=torch.float32, device=vol_bf16.device)
    _call("sceneego_unpack_volume_f32", vol_bf16, vol_bf16, C.byref(lay), batch, channels, out)
    return out


def softargmax3d(logits: torch.Tensor, multiplier: float, softmax: bool, axis: Optional[torch.Tensor],
                 coords: Optional[torch.Tensor], want_volumes: bool, out_volumes: Optional[torch.Tensor] = None):
    b, j, v = logits.shape[0], logits.shape[1], logits.shape[2]
    lib = load_library()
    ws = torch.empty(lib.sceneego_softargmax_workspace_bytes(b, j, v) // 4, dtype=torch.float32,
                     device=logits.device)
    kp = torch.empty(b, j, 3, dtype=torch.float32, device=logits.device)
    vol = None
    if want_volumes:
        vol = out_volumes if out_volumes is not None else torch.empty_like(logits)
    _call("sceneego_softargmax3d_f32", logits, logits, b, j, v, C.c_float(multiplier), int(bool(softmax)), axis, coords,
          kp, vol, ws)
    return kp, vol


# ---- backbone hand-off (SURVEY section 8f row 1) -------------------------------------------------------------
def handoff_pack(deconv_w: torch.Tensor, bn_gamma, bn_beta, bn_mean, bn_var, eps: float, conv_w: torch.Tensor,
                 conv_b: torch.Tensor, device):
    """Fold + repack the last ConvTranspose2d(256,256,4,2,1) + BatchNorm2d of pose_resnet's head and the 1x1
    process_features conv for `backbone_handoff`; returns (weights uint8 device tensor, bias f32 device tensor)."""
    import numpy as np
    lib = load_library()
    if tuple(deconv_w.shape) != (256, 256, 4, 4) or tuple(conv_w.shape[:2]) != (32, 256):
        raise SceneEgoError("handoff_pack: expects ConvTranspose2d(256,256,4) and Conv2d(256,32,1) weights")
    arrs = [t.detach().float().cpu().contiguous().numpy() for t in
            (deconv_w, bn_gamma, bn_beta, bn_mean, bn_var, conv_w.reshape(32, 256), conv_b)]
    w_out = np.zeros(lib.sceneego_handoff_weight_bytes() // 2, dtype=np.uint16)
    b_out = np.zeros(256 + 32, dtype=np.float32)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    _check(lib.sceneego_handoff_pack(ptr(arrs[0]), ptr(arrs[1]), ptr(arrs[2]), ptr(arrs[3]), ptr(arrs[4]), C.c_double(eps),
                                     ptr(arrs[5]), ptr(arrs[6]), ptr(w_out), ptr(b_out)), "handoff_pack")
    return torch.from_numpy(w_out.view(np.uint8)).to(device), torch.from_numpy(b_out).to(device)


def backbone_handoff(x: torch.Tensor, weights: torch.Tensor, bias: torch.Tensor,
                     out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x (B,256,h,w) f32 NCHW = the input of pose_resnet's last deconvolution stage -> (B,2h,2w,32) f32 channel-last,
    the stage's `feat32` (deconv + BN + ReLU + 1x1 conv fused on tcgen05; the 256-channel map is never written)."""
    b, c, h, w = x.shape
    x = x.contiguous().float()
    if out is None:
        out = torch.empty(b, 2 * h, 2 * w, 32, dtype=torch.float32, device=x.device)
    elif tuple(out.shape) != (b, 2 * h, 2 * w, 32) or out.dtype != torch.float32:
        raise SceneEgoError("backbone_handoff: bad output buffer")
    ws = torch.empty(load_library().sceneego_handoff_workspace_bytes(b, h, w), dtype=torch.uint8, device=x.device)
    _call("sceneego_backbone_handoff_f32", x, x, b, c, h, w, weights, bias, ws, out)
    return out

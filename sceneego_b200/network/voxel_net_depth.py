"""Drop-in `VoxelNetwork_depth` (reference: network/voxel_net_depth.py:19-275).

Same constructor, config keys, attributes, state-dict keys, forward signature and
4-tuple return as the reference, so `demo.py` / `test.py` can use it unchanged.
Everything after the backbone runs hand-written sm_100a kernels through the
C-ABI of include/sceneego_b200.h:

    process_features (1x1 conv; the x16 upsample + pad are never materialised
                      unless `materialize_features`)      -> sceneego_feature_conv1x1_f32
    unproject_heatmaps_one_view_batch + torch.cat         -> sceneego_unproject_f32
                          (a camera per frame, camera_ids=) -> sceneego_unproject_cameras_f32
    depth_map_to_voxel_numpy loop (host NumPy in the ref) -> sceneego_voxelize_depth_f64
                          (a camera per frame, camera_ids=) -> sceneego_voxelize_depth_cameras_f64
    point_cloud_to_voxel_numpy (clouds for scene_volumes=) -> sceneego_voxelize_points
    scan_to_voxels (world scan + B poses, scene_volumes=)   -> sceneego_voxelize_scan
    volume_net (V2VModel)                                 -> sceneego_v2v_run
    integrate_tensor_3d_with_coordinates                  -> sceneego_softargmax3d_f32

There is no CPU path: constructing on a non-CUDA device raises.
"""
import os

import numpy as np
import torch
from torch import nn

from .. import _lib
from ..utils import op
from ..utils.fisheye.FishEyeCalibrated import FishEyeCameraCalibrated
from . import pose_resnet
from .v2v import V2VModel

from .. import DEFAULT_CALIBRATION  # noqa: F401  (re-exported)

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _resolve_calibration(path):
    if os.path.exists(path):
        return path
    alt = os.path.join(_PKG, "data", os.path.basename(path))
    if os.path.exists(alt):
        return alt
    raise FileNotFoundError(path)


def _camera_model(calibration, size, n_cameras):
    """`add_camera`'s host-side checks: a calibration file path or a FishEyeCameraCalibrated whose image size is the
    module's (image_width, image_height), and room for one more camera."""
    if n_cameras >= _lib.MAX_CAMERAS:
        raise _lib.SceneEgoError(f"a module holds at most {_lib.MAX_CAMERAS} cameras")
    if isinstance(calibration, FishEyeCameraCalibrated):
        model = calibration
    elif isinstance(calibration, (str, os.PathLike)):
        model = FishEyeCameraCalibrated(calibration_file_path=_resolve_calibration(os.fspath(calibration)))
    else:
        raise _lib.SceneEgoError(f"add_camera takes a calibration file path or a FishEyeCameraCalibrated, got "
                                 f"{type(calibration).__name__}")
    got = tuple(int(v) for v in np.asarray(model.img_size).reshape(-1))
    if got != tuple(size):
        raise _lib.SceneEgoError(f"camera image size {got} differs from the module's (image_width, image_height) "
                                 f"{tuple(size)}: the feature map's crop and squash assume the module's size")
    return model


def camera_ids_host(camera_ids, b, n_cameras):
    """`camera_ids` of lift() / forward() -> (B,) int32 NumPy array.  Host-side only (a list, a NumPy array or a CPU
    tensor of integers): ids on the device could only be checked after a synchronisation."""
    if isinstance(camera_ids, torch.Tensor):
        if camera_ids.device.type != "cpu":
            raise _lib.SceneEgoError("camera_ids must be a host-side sequence (list, NumPy array or CPU tensor), got a "
                                     f"tensor on {camera_ids.device}: checking device ids would need a synchronisation")
        if camera_ids.dtype == torch.bool or camera_ids.dtype.is_floating_point or camera_ids.dtype.is_complex:
            raise _lib.SceneEgoError(f"camera_ids must be integers, got {camera_ids.dtype}")
        a = camera_ids.numpy()
    else:
        a = np.asarray(camera_ids)
    if a.dtype.kind not in "iu":
        raise _lib.SceneEgoError(f"camera_ids must be integers, got {a.dtype}")
    if a.shape != (b,):
        raise _lib.SceneEgoError(f"camera_ids must hold one id per frame ({b}), got shape {a.shape}")
    if a.min() < 0 or a.max() >= n_cameras:
        raise _lib.SceneEgoError(f"camera_ids must lie in [0, {n_cameras}) (cameras come from add_camera), got "
                                 f"[{a.min()}, {a.max()}]")
    return a.astype(np.int32)


def camera_frame_order(ids):
    """Stable sort of the frames by camera: the order the camera-per-frame kernels visit frames in, so that frames
    that share a camera are adjacent and a voxel's geometry (a pixel's ray) is reloaded once per run."""
    return np.argsort(np.asarray(ids), kind="stable").astype(np.int32)


class VoxelNetwork_depth(nn.Module):
    def __init__(self, config, device='cuda', materialize_features=True, materialize_volumes=True,
                 fused_projection=False, v2v_chunk=32, persistent_features=False, graph_max_batch=0,
                 backbone_handoff=False, act_dtype=None):
        """Extra keyword switches (all default to reference-identical outputs):
        materialize_features / materialize_volumes: build outputs #2 / #3 of the reference
            forward (168 MB and 15.7 MB per frame, ignored by demo.py:57 / test.py:54);
            False returns None in their place.
        fused_projection: project voxel centres inside the gather kernel (Scaramuzza in-kernel)
            instead of reading the `grid_coord_proj_batch` argument.
        persistent_features: output #2 is a view of ONE buffer that the next call overwrites (default: a fresh
            tensor per call, like the reference).
        graph_max_batch: batches of at most this many frames replay a captured CUDA graph of the whole lift
            (demo.py runs batch 1: ~70 launches of a few microseconds each are launch-bound otherwise); 0 = off.
        backbone_handoff: forward() fuses the backbone's last deconvolution stage (ConvTranspose2d + BN + ReLU) with
            process_features[0] in one tensor-core kernel (bf16 operands, fp32 accumulation) instead of running the
            stage in torch and the 1x1 conv in fp32; `lift()` is unaffected.
        act_dtype: "bf16" (default) or "f16" -- storage type of the V2V activations and packed weights.  "f16" loads
            libsceneego_b200_f16.so (same kernels, IEEE fp16 cells with saturating stores): same speed, 8-9x smaller
            storage-rounding error (33.9 -> 3.7 mm in the sharp-softmax test).  One dtype per process."""
        super().__init__()
        dev = torch.device(device)
        if dev.type != 'cuda':
            raise _lib.SceneEgoError("sceneego_b200.VoxelNetwork_depth needs a CUDA device (no CPU fallback)")
        if act_dtype is not None:
            _lib.set_act_dtype(act_dtype)
        _lib.load_library()
        dev = _lib._as_device(dev)
        self.device = device
        self.persistent_features = persistent_features
        self.backbone_handoff = bool(backbone_handoff)
        self._handoff_cache = None
        self.graph_max_batch = int(graph_max_batch)
        self._graphs = {} if graph_max_batch > 0 else None
        self.num_joints = config.model.backbone.num_joints
        self.volume_softmax = config.model.volume_softmax
        self.volume_multiplier = config.model.volume_multiplier
        self.volume_size = config.model.volume_size
        self.cuboid_side = config.model.cuboid_side
        self.kind = config.model.kind
        self.heatmap_softmax = config.model.heatmap_softmax
        self.heatmap_multiplier = config.model.heatmap_multiplier
        self.materialize_features = materialize_features
        self.materialize_volumes = materialize_volumes
        self.fused_projection = fused_projection

        if config.model.backbone.local_checkpoint:
            loads = torch.load(config.model.backbone.checkpoint)
            self.backbone = pose_resnet.get_pose_net(state_dict=loads['state_dict'])
        else:
            print('Do not load checkpoint')
            self.backbone = pose_resnet.get_pose_net(None)
        self.backbone = self.backbone.to(device)
        if config.opt.train_2d is False:
            for p in self.backbone.parameters():
                p.requires_grad = False

        self.heatmap_shape = tuple(config.heatmap_shape)                     # (1024, 1280)
        self.image_width = config.dataset.image_width
        self.image_height = config.dataset.image_height
        # parameter container only (state-dict keys process_features.0.{weight,bias});
        # the Upsample / ConstantPad2d children hold no parameters
        self.process_features = nn.Sequential(
            nn.Conv2d(256, 32, 1),
            nn.Upsample(size=(self.image_height, self.image_height)),
            nn.ConstantPad2d(padding=((self.image_width - self.image_height) // 2,
                                      (self.image_width - self.image_height) // 2, 0, 0), value=0.0),
        ).to(device)

        self.with_scene = config.model.with_scene
        self.with_intersection = False
        if self.with_scene is True:
            if config.model.with_intersection is True:
                volume_input_channel_num = 32 + 1 + 32       # volumes, volumes * scene, scene (:66-68, :257-260)
                self.with_intersection = True
            else:
                volume_input_channel_num = 32 + 1
                self.with_intersection = False
        else:
            volume_input_channel_num = 32
        self.volume_net = V2VModel(volume_input_channel_num, self.num_joints, max_chunk=v2v_chunk).to(device)

        print('build coord volume')
        self.fisheye_camera_model = FishEyeCameraCalibrated(
            calibration_file_path=_resolve_calibration(config.dataset.camera_calibration_path))
        self._calib = self.fisheye_camera_model.calib_struct(self.image_width, self.image_height)
        self.coord_volume = self.build_coord_volume()
        self.coord_volumes = self.coord_volume.unsqueeze(0).expand(config.opt.batch_size, -1, -1, -1, -1)
        print('build reprojected grid coord')
        self.grid_coord_proj = op.get_projected_2d_points_with_coord_volumes(
            fisheye_model=self.fisheye_camera_model, coord_volume=self.coord_volume)
        self.grid_coord_proj_batch = op.get_grid_coord_proj_batch(
            self.grid_coord_proj, batch_size=config.opt.batch_size, heatmap_shape=config.heatmap_shape)
        # ray table: device copy row-major for the kernel, NumPy x-major copy for API parity
        self._ray_dev = self.fisheye_camera_model.ray_table_device(self.image_width, self.image_height, dev)
        self.ray = self._ray_dev.permute(1, 0, 2).reshape(-1, 3).cpu().numpy()
        # cameras for camera_ids= (add_camera); camera 0 is the config's.  The stacked (K,N,2) grids and
        # (K,H,W,3) ray tables are built when first needed and rebuilt (new storage) by add_camera
        self.cameras = [self.fisheye_camera_model]
        self._cam_calibs = [self._calib]
        self._cam_grids = None
        self._cam_rays = None
        cv = self.coord_volume
        self._axis = torch.stack([cv[:, 0, 0, 0], cv[0, :, 0, 1], cv[0, 0, :, 2]]).contiguous()
        self.last_launches = 0
        self._side_streams = {}
        self._features_buf = None
        self._grid_checked = None
        self._coord_checked = None
        self.keep_logits = False     # True: the V2V logits of the last call stay in `last_logits` (tests, diagnostics)
        self.last_logits = None
        # (pre_h, pre_w, clamp_max): depth_map_batch holds RAW decoded maps and the dataset's preprocessing
        # (dataset/demo_dataset.py:86-91: nearest resize to 1280x1024, depth > 10 -> 10) is fused into the
        # voxelisation kernel's load; None: the caller has preprocessed them, like the reference's datasets do
        self.depth_preprocess = None

    def build_coord_volume(self):
        """network/voxel_net_depth.py:110-134, on the device (fp32, mul then add)."""
        v, s = self.volume_size, self.cuboid_side
        idx = torch.arange(v, dtype=torch.float32, device=self.device)
        step = float(s / (v - 1))
        axy = float(-s / 2) + step * idx
        az = 0.0 + step * idx
        gx, gy, gz = torch.meshgrid(axy, axy, az, indexing='ij')
        return torch.stack([gx, gy, gz], dim=-1).contiguous()

    # ------------------------------------------------------------------ cameras
    def add_camera(self, calibration) -> int:
        """Set up one more fisheye camera for `camera_ids=` and return its id.  `calibration` is a calibration file path
        or a FishEyeCameraCalibrated of the module's image size.  Its calib struct, table-mode grid and ray table are
        built by the functions the constructor uses, so frames of this camera lift exactly as they would through a
        module built from that file.  The reference attributes (ray, grid_coord_proj_batch, ...) stay camera 0's."""
        model = _camera_model(calibration, (self.image_width, self.image_height), len(self.cameras))
        dev = _lib._as_device(self.device)
        grid_px = op.get_projected_2d_points_with_coord_volumes(fisheye_model=model, coord_volume=self.coord_volume)
        grid = op.get_grid_coord_proj_batch(grid_px, batch_size=1, heatmap_shape=self.heatmap_shape)
        grid = grid[0].reshape(-1, 2).contiguous().float()
        ray = model.ray_table_device(self.image_width, self.image_height, dev)
        grids, rays = self._camera_tables()
        self._cam_grids = torch.cat([grids, grid.unsqueeze(0)])
        self._cam_rays = torch.cat([rays, ray.unsqueeze(0)])
        self._cam_calibs.append(model.calib_struct(self.image_width, self.image_height))
        self.cameras.append(model)
        return len(self.cameras) - 1

    def _camera_tables(self):
        """(K,N,2) f32 table-mode grids and (K,H,W,3) fp64 ray tables of the cameras, camera 0 first."""
        if self._cam_grids is None:
            self._cam_grids = self._grid_table(self.grid_coord_proj_batch, 1).unsqueeze(0)
            self._cam_rays = self._ray_dev.unsqueeze(0)
        return self._cam_grids, self._cam_rays

    def _camera_ids(self, camera_ids, grid_coord_proj_batch, b):
        """Checked host ids, or None.  Per-camera grids come from add_camera, so the grid argument must be the
        module's own table."""
        if camera_ids is None:
            return None
        ids = camera_ids_host(camera_ids, b, len(self.cameras))
        own, g = self.grid_coord_proj_batch, grid_coord_proj_batch
        if g is not own and not (isinstance(g, torch.Tensor) and g.dtype == own.dtype and g.device == own.device
                                 and g.data_ptr() == own.data_ptr() and g.shape[1:] == own.shape[1:]
                                 and g.stride() == own.stride()):
            raise _lib.SceneEgoError("with camera_ids, grid_coord_proj_batch must be the module's own table: the "
                                     "per-camera tables come from add_camera")
        self._camera_tables()
        return ids

    @staticmethod
    def _camera_host(ids, chunk):
        """ids and, per V2V chunk, the chunk's stable frame order (chunk-local indices) as one pinned (2B,) int32
        tensor [ids | order], so that its copy to the device needs no synchronisation."""
        b = ids.shape[0]
        h = torch.empty(2 * b, dtype=torch.int32, pin_memory=True)
        h.numpy()[:b] = ids
        h.numpy()[b:] = np.concatenate([camera_frame_order(ids[s:s + chunk]) for s in range(0, b, chunk)])
        return h

    # ------------------------------------------------------------------ argument handling
    def _grid_table(self, grid_coord_proj_batch, b):
        """(>=B, N, 1, 2) normalised projection grid -> the (N, 2) table the gather kernel reads.  The reference
        slices the argument to the batch (:241-242) and samples frame i with row i; its callers always pass the
        batch-expanded (stride-0) table of the module.  A materialised copy is accepted when all rows are equal."""
        g = grid_coord_proj_batch
        n = self.volume_size ** 3
        if g.dim() != 4 or tuple(g.shape[1:]) != (n, 1, 2) or g.shape[0] < 1:
            raise _lib.SceneEgoError(f"grid_coord_proj_batch must have shape (>=B, {n}, 1, 2), got {tuple(g.shape)}")
        expanded = g.shape[0] == 1 or g.stride(0) == 0        # one table for every frame: any batch size is fine
        if g.shape[0] < b and not expanded:
            raise _lib.SceneEgoError("grid_coord_proj_batch holds fewer rows than the batch (the reference fails "
                                     "in F.grid_sample here, utils/op.py:209)")
        if not expanded:
            key = (g.data_ptr(), g._version, tuple(g.shape), b)
            if key != self._grid_checked:
                if not bool((g[:b] == g[:1]).all()):
                    raise _lib.SceneEgoError("per-frame projection grids are not supported (the reference expands "
                                             "one table, utils/op.py:177-184)")
                self._grid_checked = key
        return g[0].reshape(-1, 2).contiguous().float()

    def _coord_table(self, coord_volumes, b):
        """None / the module's own table -> None (the kernel uses the three per-axis tables of `coord_volume`);
        any other (>=B, V, V, V, 3) tensor is honoured: its first row becomes the (N, 3) coordinate table the
        soft-argmax multiplies with, like utils/op.py:94 does."""
        if coord_volumes is None:
            return None
        c, v = coord_volumes, self.volume_size
        expanded = c.dim() == 5 and (c.shape[0] == 1 or c.stride(0) == 0)
        if c.dim() != 5 or tuple(c.shape[1:]) != (v, v, v, 3) or (c.shape[0] < b and not expanded):
            raise _lib.SceneEgoError(f"coord_volumes must have shape (>=B, {v}, {v}, {v}, 3), got {tuple(c.shape)}")
        if c.data_ptr() == self.coord_volume.data_ptr() and c.dtype == self.coord_volume.dtype:
            return None
        if not expanded:
            key = (c.data_ptr(), c._version, tuple(c.shape), b)
            if key != self._coord_checked:
                if not bool((c[:b] == c[:1]).all()):
                    raise _lib.SceneEgoError("per-frame coordinate volumes are not supported (the reference expands "
                                             "one table, network/voxel_net_depth.py:81-83)")
                self._coord_checked = key
        return c[0].reshape(-1, 3).contiguous().float()

    # ------------------------------------------------------------------ hot path
    def lift(self, backbone_features, grid_coord_proj_batch, coord_volumes=None, scene_volumes=None,
             depth_map_batch=None, camera_ids=None):
        """Everything the reference forward does after `self.backbone(images)`
        (network/voxel_net_depth.py:237-273).  camera_ids: None (every frame through camera 0, the config's), or one
        camera id per frame (a list, NumPy array or CPU tensor of ints in [0, len(self.cameras))): frame b is lifted
        exactly as a module built from camera camera_ids[b]'s calibration would lift it in the same batch."""
        if self.training:
            raise _lib.SceneEgoError("VoxelNetwork_depth is inference-only (BatchNorm is folded from the running "
                                     "statistics): call .eval() first, like demo.py:32 / test.py:29")
        feat = backbone_features.contiguous().float()
        if not feat.is_cuda:
            raise _lib.SceneEgoError("sceneego_b200 ops need CUDA tensors (no CPU fallback)")
        conv = self.process_features[0]
        return self._lift_feat32(lambda out: _lib.feature_conv1x1(feat, conv.weight, conv.bias, out=out),
                                 feat.shape[0], (feat.shape[2], feat.shape[3]), feat.device, 1,
                                 grid_coord_proj_batch, coord_volumes, scene_volumes, depth_map_batch, camera_ids)

    def _lift_feat32(self, make_feat32, b, hw, dev, feat_launches, grid_coord_proj_batch, coord_volumes, scene_volumes,
                     depth_map_batch, camera_ids=None):
        """The stage from `feat32` on.  `make_feat32(out)` produces the (B,h,w,32) channel-last f32 map of
        process_features[0] -- from the backbone's 256-channel features (lift) or fused with the backbone's last
        deconvolution (forward with backbone_handoff=True) -- into `out` (None: a fresh tensor)."""
        v = self.volume_size
        ids = self._camera_ids(camera_ids, grid_coord_proj_batch, b)
        if b <= self.graph_max_batch and self._graphs is not None:
            out = self._lift_graphed(make_feat32, b, hw, dev, feat_launches, grid_coord_proj_batch, coord_volumes,
                                     scene_volumes, depth_map_batch, ids)
            if out is not NotImplemented:
                return out
        feat32 = make_feat32(None)                                            # (B,64,64,32) channel-last
        launches = feat_launches
        features = None
        feat_done = None
        main = torch.cuda.current_stream(dev)
        if self.materialize_features:
            # output #2 of the reference is a pure HBM write (168 MB/frame) nothing downstream reads: it runs on a
            # side stream and shares the SMs (and the idle HBM bandwidth) with the tensor-bound V2V kernels.
            # The tensor is FRESH per call, like the reference's (`persistent_features=True` reuses one buffer that
            # the next call overwrites).  It is allocated on, and at the end of lift() re-joined to, the current
            # stream (wait_event below), so the caching allocator's usual stream-ordered reuse is correct without
            # record_stream -- which is what made freed 10 GB blocks pile up in round 1.
            side = self._side_streams.get(dev)
            if side is None:
                side = self._side_streams[dev] = torch.cuda.Stream(device=dev)
            shape = (b, 32, self.image_height, self.image_width)
            if self.persistent_features:
                buf = self._features_buf
                if buf is None or buf.device != dev or buf.shape[0] < b:
                    self._features_buf = buf = None
                    self._features_buf = buf = torch.empty(shape, dtype=torch.float32, device=dev)
                features = buf[:b]
            else:
                features = torch.empty(shape, dtype=torch.float32, device=dev)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                _lib.features_upsample_pad(feat32, self.image_height, (self.image_width - self.image_height) // 2,
                                           out=features)
                feat_done = torch.cuda.Event()
                feat_done.record(side)
            launches += 1
        if self.with_scene is True and scene_volumes is None and depth_map_batch is None:
            print("no scene volume or depth input!")
            if feat_done is not None:
                main.wait_event(feat_done)
            return None
        grid = None if self.fused_projection else self._grid_table(grid_coord_proj_batch, b)
        coords = self._coord_table(coord_volumes, b)
        vn = self.volume_net
        pg = vn.program(v, min(vn.max_chunk, b), dev)
        chunk = pg.chunk
        cam = None if ids is None else self._camera_host(ids, chunk).to(dev, non_blocking=True)
        logits = torch.empty(b, self.num_joints, v, v, v, dtype=torch.float32, device=dev)
        for s in range(0, b, chunk):
            n = min(chunk, b - s)
            launches += self._fill_v2v_input(pg, feat32[s:s + n], grid,
                                             None if scene_volumes is None else scene_volumes[s:s + n],
                                             None if depth_map_batch is None else depth_map_batch[s:s + n],
                                             None if cam is None else (cam[s:s + n], cam[b + s:b + s + n]))
            launches += vn.run_chunk(pg, n, logits[s:s + n])
        kp, volumes = _lib.softargmax3d(logits, float(self.volume_multiplier), bool(self.volume_softmax),
                                        self._axis if coords is None else None, coords, self.materialize_volumes)
        launches += 3 if self.materialize_volumes else 2
        if feat_done is not None:
            main.wait_event(feat_done)
        self.last_launches = launches
        self.last_logits = logits if self.keep_logits else None
        return kp, features, volumes, self.coord_volumes

    def _lift_graphed(self, make_feat32, b, hw, dev, feat_launches, grid_coord_proj_batch, coord_volumes, scene_volumes,
                      depth_map_batch, ids=None):
        """Small batches (demo.py runs batch 1): the ~68 launches from the gather to the V2V logits replay as ONE
        captured CUDA graph over static buffers; the 1x1 feature conv (live weights), the copy of the scene input
        into its static buffer, the soft-argmax and outputs #2 / #3 (fresh tensors) stay outside the graph.
        Returns NotImplemented when the eager path must handle the call."""
        if self.with_scene is True and scene_volumes is None and depth_map_batch is None:
            return NotImplemented
        v = self.volume_size
        vn = self.volume_net
        if min(vn.max_chunk, self.graph_max_batch) < b:
            return NotImplemented
        grid = None if self.fused_projection else self._grid_table(grid_coord_proj_batch, b)
        coords = self._coord_table(coord_volumes, b)
        pg = vn.program(v, min(vn.max_chunk, self.graph_max_batch), dev)
        src, kind = None, "none"
        if self.with_scene is True:
            kind = "scene" if scene_volumes is not None else "depth"
            src = scene_volumes if scene_volumes is not None else depth_map_batch
            src = src.reshape((b,) + tuple(src.shape[-3:] if kind == "scene" else src.shape[-2:]))
            if kind == "scene" and self.with_intersection:
                return NotImplemented                       # the eager path raises the explanatory error
        # camera mode: the ids and frame order live in a static buffer refilled before every replay, so a new
        # assignment replays the same capture; add_camera reallocates the stacked tables, which recaptures
        cams = None if ids is None else (self._cam_grids.data_ptr(), self._cam_rays.data_ptr())
        key = (b, kind, None if src is None else tuple(src.shape), bool(self.fused_projection),
               0 if grid is None else grid.data_ptr(), self.depth_preprocess, id(pg), dev.index, cams)
        g = self._graphs.get(key)
        main = torch.cuda.current_stream(dev)
        if g is None:
            if len(self._graphs) >= 8 or any(e["pg"] is not pg for e in self._graphs.values()):
                self._graphs.clear()                        # a rebuilt program (new weights) invalidates every capture
            g = {"pg": pg, "grid": grid,
                 "feat32": torch.empty(b, hw[0], hw[1], 32, dtype=torch.float32, device=dev),
                 "src": None if src is None else torch.empty(src.shape, dtype=torch.float32, device=dev),
                 "logits": torch.empty(b, self.num_joints, v, v, v, dtype=torch.float32, device=dev),
                 "cam": None if ids is None else torch.empty(2 * b, dtype=torch.int32, device=dev)}

            def body():
                n = self._fill_v2v_input(pg, g["feat32"], grid, g["src"] if kind == "scene" else None,
                                         g["src"] if kind == "depth" else None,
                                         None if ids is None else (g["cam"][:b], g["cam"][b:]))
                return n + vn.run_chunk(pg, b, g["logits"])
            make_feat32(g["feat32"])
            if src is not None:
                g["src"].copy_(src)
            if ids is not None:
                g["cam"].copy_(self._camera_host(ids, b), non_blocking=True)
            body()                                          # eager warm-up: per-device kernel attributes get set
            main.synchronize()
            graph = torch.cuda.CUDAGraph()
            with _lib.on_device(dev), torch.cuda.graph(graph):
                g["launches"] = body()
            g["graph"] = graph
            self._graphs[key] = g
        make_feat32(g["feat32"])
        if src is not None:
            g["src"].copy_(src)
        if ids is not None:
            g["cam"].copy_(self._camera_host(ids, b), non_blocking=True)
        features, feat_done = None, None
        if self.materialize_features:
            side = self._side_streams.get(dev)
            if side is None:
                side = self._side_streams[dev] = torch.cuda.Stream(device=dev)
            features = torch.empty(b, 32, self.image_height, self.image_width, dtype=torch.float32, device=dev)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                _lib.features_upsample_pad(g["feat32"], self.image_height,
                                           (self.image_width - self.image_height) // 2, out=features)
                feat_done = torch.cuda.Event()
                feat_done.record(side)
        g["graph"].replay()
        kp, volumes = _lib.softargmax3d(g["logits"], float(self.volume_multiplier), bool(self.volume_softmax),
                                        self._axis if coords is None else None, coords, self.materialize_volumes)
        if feat_done is not None:
            main.wait_event(feat_done)
        self.last_launches = feat_launches + g["launches"] + (3 if self.materialize_volumes else 2) + (1 if features is not None else 0)
        self.last_logits = g["logits"].clone() if self.keep_logits else None
        return kp, features, volumes, self.coord_volumes

    def _fill_v2v_input(self, pg, feat32, grid, scene_volumes, depth_map_batch, cams=None) -> int:
        """a2 + a5 + a6: write the lifted features and the scene occupancy of `n` frames straight into the V2V
        program's input buffer (network/voxel_net_depth.py:243-262).  cams: None (camera 0) or the (n,) int32 device
        camera ids and chunk-local frame order of the frames.  Returns the number of kernels launched."""
        n = feat32.shape[0]
        v = self.volume_size
        in_buf = pg.buffers[pg.in_buf]
        img_h, img_w = self.heatmap_shape
        if cams is None:
            _lib.unproject(feat32, grid, self._calib if self.fused_projection else None, v, float(self.cuboid_side),
                           img_h, img_w, None, in_buf, pg.lay_in, extra_zero_planes=pg.extra_zero_planes)
        else:
            _lib.unproject_cameras(feat32, None if self.fused_projection else self._cam_grids, self._cam_calibs, cams[0],
                                   cams[1], v, float(self.cuboid_side), img_h, img_w, None, in_buf, pg.lay_in,
                                   extra_zero_planes=pg.extra_zero_planes)
        launches = 1
        if self.with_scene is True:
            scene_ch = 64 if self.with_intersection else 32
            if scene_volumes is not None:
                if self.with_intersection:
                    # the reference concatenates 33 channels here and its 65-channel V2V then fails (:246-249)
                    raise _lib.SceneEgoError("with_intersection=true takes depth_map_batch, not scene_volumes "
                                             "(the reference builds a 33-channel input on this path)")
                sv = scene_volumes.contiguous().float().unsqueeze(1)
                _lib.pack_volume(sv, in_buf, pg.lay_in, c_offset=32)
            else:
                d = depth_map_batch
                d = d.reshape(n, d.shape[-2], d.shape[-1]).contiguous().float()
                # z-window input (the marching stem): one store per pixel into the program's plain f32 grid, then
                # one pass builds the whole occupancy plane from it and leaves the grid zero for the next batch
                scratch = pg.occ_scratch[:n] if pg.zwin else None
                dst_bf16 = None if pg.zwin else in_buf
                if cams is not None:
                    pre, cm = (None, float("inf")) if self.depth_preprocess is None else \
                        (self.depth_preprocess[:2], float(self.depth_preprocess[2]))
                    _lib.voxelize_depth_cameras(d, pre, cm, self._cam_rays, cams[0], cams[1], self.image_height,
                                                self.image_width, v, float(self.cuboid_side), scratch, dst_bf16,
                                                pg.lay_in, channel=scene_ch)
                elif self.depth_preprocess is not None:
                    ph, pw, cm = self.depth_preprocess
                    _lib.voxelize_depth_raw(d, (ph, pw), float(cm), self._ray_dev, self.image_height,
                                            self.image_width, v, float(self.cuboid_side), scratch, dst_bf16, pg.lay_in,
                                            channel=scene_ch)
                else:
                    _lib.voxelize_depth(d, self._ray_dev, self.image_height, self.image_width, v,
                                        float(self.cuboid_side), scratch, dst_bf16, pg.lay_in, channel=scene_ch)
                if pg.zwin:
                    _lib.occ_expand_zwin(scratch, in_buf, pg.lay_in, scene_ch)
                    launches += 1
                if self.with_intersection:
                    _lib.intersect(in_buf, pg.lay_in, n, 32)
                    launches += 1
            launches += 1
        return launches

    def forward(self, images, grid_coord_proj_batch, coord_volumes, scene_volumes=None, depth_map_batch=None,
                camera_ids=None):
        if self.backbone_handoff:
            # SURVEY section 8f row 1: the backbone stops before its last deconvolution stage; that stage, its
            # BatchNorm + ReLU and process_features[0] run as ONE tcgen05 kernel that emits the stage's channel-last
            # feat32 directly (the heatmap head `final_layer`, unused by the reference forward, is skipped)
            if self.training:
                raise _lib.SceneEgoError("VoxelNetwork_depth is inference-only: call .eval() first")
            x2 = self.backbone.forward_before_last_deconv(images).contiguous().float()
            w, bias = self._handoff_weights(x2.device)
            return self._lift_feat32(lambda out: _lib.backbone_handoff(x2, w, bias, out=out), x2.shape[0],
                                     (2 * x2.shape[2], 2 * x2.shape[3]), x2.device, 2, grid_coord_proj_batch,
                                     coord_volumes, scene_volumes, depth_map_batch, camera_ids)
        heatmaps, features = self.backbone(images)
        return self.lift(features, grid_coord_proj_batch, coord_volumes, scene_volumes, depth_map_batch, camera_ids)

    def _handoff_weights(self, device):
        """Packed weights of the hand-off kernel, rebuilt when one of their sources changed (in-place edits bump
        `_version`, .to()/load_state_dict(assign=True) change the storage)."""
        dc, bn, pf = self.backbone.deconv_layers[6], self.backbone.deconv_layers[7], self.process_features[0]
        src = (dc.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var, pf.weight, pf.bias)
        key = tuple((t.data_ptr(), t._version) for t in src) + (str(device),)
        if self._handoff_cache is None or self._handoff_cache[0] != key:
            w, bias = _lib.handoff_pack(dc.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var, float(bn.eps),
                                        pf.weight, pf.bias, device)
            self._handoff_cache = (key, w, bias)
        return self._handoff_cache[1], self._handoff_cache[2]

    # kept for API parity with the reference (network/voxel_net_depth.py:194-205): one frame
    def depth_map_to_voxel_numpy(self, depth):
        d = depth.reshape(1, depth.shape[-2], depth.shape[-1]).contiguous().float().to(self.device)
        occ = torch.zeros(1, self.volume_size, self.volume_size, self.volume_size, dtype=torch.float32,
                          device=d.device)
        _lib.voxelize_depth(d, self._ray_dev, self.image_height, self.image_width, self.volume_size,
                            float(self.cuboid_side), occ, None, None)
        return occ[0]

    def point_cloud_to_voxel_numpy(self, scene_point_cloud):
        """network/voxel_net_depth.py:207-222: one camera-space (N,3) cloud -- NumPy array or torch tensor, CPU (copied
        to the module's device once) or CUDA -> (V,V,V) f32 {0,1} on the module's device, with the module's
        `volume_size` and `cuboid_side`.  A float64 cloud is quantised in fp64 (what depth_map_to_voxel_numpy builds:
        fp64 rays times depth), a float32 one in fp32, like NumPy.  Stack the grids of a batch and pass them as
        `scene_volumes=`."""
        p = torch.as_tensor(scene_point_cloud).reshape(-1, 3)
        dev = _lib._as_device(self.device)
        if p.device != dev:
            p = p.to(dev)
        occ = torch.zeros(1, self.volume_size, self.volume_size, self.volume_size, dtype=torch.float32, device=dev)
        _lib.voxelize_points(p.contiguous(), torch.tensor([0, p.shape[0]], dtype=torch.int64), self.volume_size,
                             float(self.cuboid_side), occ)
        return occ[0]

    def scan_to_voxels(self, scan, cam_from_world):
        """One static world-space (N,3) scan and B (4,4) cam_from_world poses -- NumPy arrays or torch tensors, CPU
        (the scan is copied to the module's device) or CUDA -> (B,V,V,V) f32 {0,1} on the module's device, with the
        module's `volume_size` and `cuboid_side`, in one launch (sceneego_voxelize_scan).  Frame b's grid is
        point_cloud_to_voxel_numpy of the scan mapped into camera b's frame (the frame of ray x depth) by
        `A[k,0]*x + A[k,1]*y + A[k,2]*z + t[k]` in the scan's precision; the poses must have the scan's dtype.
        Pass the result as `scene_volumes=`."""
        p = torch.as_tensor(scan)
        dev = _lib._as_device(self.device)
        if p.device != dev:
            p = p.to(dev)
        v = self.volume_size
        pose = torch.as_tensor(cam_from_world)
        occ = torch.zeros(pose.shape[0] if pose.dim() == 3 else 0, v, v, v, dtype=torch.float32, device=dev)
        _lib.voxelize_scan(p.contiguous(), pose, v, float(self.cuboid_side), occ)
        return occ

    def calculated_ray_direction_numpy(self, image_width, image_height):
        """network/voxel_net_depth.py:147-155: the (W*H, 3) fp64 unit-ray table in the reference's x-major order
        (row x*H + y), computed on the device (sceneego_ray_table_f64) and copied to the host as a NumPy array."""
        ray = self.fisheye_camera_model.ray_table_device(image_width, image_height, _lib._as_device(self.device))
        return ray.permute(1, 0, 2).reshape(-1, 3).cpu().numpy()

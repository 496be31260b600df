"""Deterministic synthetic inputs and weights (SURVEY.md section 8d).

No checkpoint or dataset is available offline, so tests and the benchmark use
seeded synthetic data.  Weights are generated per state-dict key from a
generator seeded by crc32(key), so two modules with the same key set (the
reference's and ours) get identical values regardless of construction order.
"""
from __future__ import annotations

import math
import zlib
from typing import Dict, Iterable, Tuple

import numpy as np
import torch


def _gen(key: str, seed: int) -> torch.Generator:
    g = torch.Generator(device="cpu")
    g.manual_seed((zlib.crc32(key.encode()) ^ (seed * 0x9E3779B1)) & 0x7FFFFFFF)
    return g


def synthetic_state_dict(shapes: Iterable[Tuple[str, Tuple[int, ...]]], seed: int = 0,
                         mode: str = "random_bn", logit_scale: float = 1.0) -> Dict[str, torch.Tensor]:
    """mode 'default' mimics the reference init (xavier_normal_ convs, zero
    bias, identity BatchNorm -- network/v2v.py:172-181); mode 'random_bn'
    randomises biases and BatchNorm statistics so that BN folding is exercised.
    `logit_scale` multiplies volume_net.output_layer to sharpen the softmax.
    """
    sd = {}
    for key, shape in shapes:
        shape = tuple(shape)
        g = _gen(key, seed)
        leaf = key.rsplit(".", 1)[-1]
        if leaf == "num_batches_tracked":
            t = torch.zeros((), dtype=torch.long)
        elif len(shape) >= 3:  # conv / deconv weight
            rf = int(np.prod(shape[2:]))
            std = math.sqrt(2.0 / ((shape[0] + shape[1]) * rf))
            t = torch.randn(shape, generator=g) * std
        elif leaf == "running_mean":
            t = torch.randn(shape, generator=g) * 0.1 if mode == "random_bn" else torch.zeros(shape)
        elif leaf == "running_var":
            t = torch.rand(shape, generator=g) * 1.5 + 0.5 if mode == "random_bn" else torch.ones(shape)
        elif leaf == "weight":  # BatchNorm gamma
            t = torch.rand(shape, generator=g) + 0.5 if mode == "random_bn" else torch.ones(shape)
        elif leaf == "bias":
            t = torch.randn(shape, generator=g) * 0.1 if mode == "random_bn" else torch.zeros(shape)
        else:
            raise KeyError(key)
        if logit_scale != 1.0 and key.endswith("volume_net.output_layer.weight"):
            t = t * logit_scale
        sd[key] = t
    return sd


def synthetic_features(batch: int, seed: int = 1234, hw: int = 64, channels: int = 256) -> torch.Tensor:
    """Backbone-like post-ReLU features (B,256,64,64) f32."""
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    return torch.relu(torch.randn(batch, channels, hw, hw, generator=g))


def synthetic_depth_uniform(batch: int, seed: int = 42, h: int = 1024, w: int = 1280, hi: float = 4.0
                            ) -> torch.Tensor:
    """Dense-scatter stress: U(0, hi) metres."""
    rng = np.random.default_rng(seed)
    return torch.from_numpy((rng.random((batch, h, w), dtype=np.float32) * np.float32(hi)))


def synthetic_depth_room(batch: int, ray: np.ndarray, seed: int = 7, h: int = 1024, w: int = 1280,
                         clamp: float = 10.0) -> torch.Tensor:
    """Real-like depth: range to the walls of an axis-aligned room around the
    head-mounted camera, zero outside the r<=512 px image circle, clamped at
    `clamp` metres like dataset/demo_dataset.py:91.  `ray` is the (w*h,3)
    x-major unit-ray table."""
    rng = np.random.default_rng(seed)
    r = ray.reshape(w, h, 3).transpose(1, 0, 2)  # (h, w, 3)
    out = np.zeros((batch, h, w), dtype=np.float32)
    yy, xx = np.mgrid[0:h, 0:w]
    circle = (xx - w / 2) ** 2 + (yy - h / 2) ** 2 <= 512 ** 2
    for b in range(batch):
        half = np.array([rng.uniform(1.0, 2.5), rng.uniform(1.0, 2.5)])
        floor = rng.uniform(1.2, 1.8)
        with np.errstate(divide="ignore", invalid="ignore"):
            tx = np.where(r[..., 0] != 0, half[0] / np.abs(r[..., 0]), np.inf)
            ty = np.where(r[..., 1] != 0, half[1] / np.abs(r[..., 1]), np.inf)
            tz = np.where(r[..., 2] > 0, floor / r[..., 2], np.inf)
        t = np.minimum(np.minimum(tx, ty), tz)
        t = np.where(np.isfinite(t), t, clamp)
        out[b] = np.where(circle, np.minimum(t, clamp), 0.0).astype(np.float32)
    return torch.from_numpy(out)


ROOM_SIZE = (10.0, 8.0, 3.0)      # synthetic_world_scan's room: x, y extent of the floor and the height, metres


def synthetic_world_scan(n: int, seed: int = 0, dtype=np.float64) -> np.ndarray:
    """A static world-space scan like a mesh, SLAM map or LiDAR sweep would give: n points sampled uniformly by area
    from the floor (z = 0), the four walls and the ceiling of a ROOM_SIZE room, and the five visible faces of four
    boxes standing on the floor, with 5 mm of noise.  World z points up.  (n,3) in `dtype`."""
    rng = np.random.default_rng(seed)
    W, D, H = ROOM_SIZE
    # axis-aligned rectangles: (origin, edge u, edge v)
    rects = [((0, 0, 0), (W, 0, 0), (0, D, 0)), ((0, 0, H), (W, 0, 0), (0, D, 0)),
             ((0, 0, 0), (W, 0, 0), (0, 0, H)), ((0, D, 0), (W, 0, 0), (0, 0, H)),
             ((0, 0, 0), (0, D, 0), (0, 0, H)), ((W, 0, 0), (0, D, 0), (0, 0, H))]
    for _ in range(4):
        sx, sy, sz = rng.uniform(0.4, 1.2), rng.uniform(0.4, 1.2), rng.uniform(0.3, 1.0)
        ox, oy = rng.uniform(0.5, W - 0.5 - sx), rng.uniform(0.5, D - 0.5 - sy)
        rects += [((ox, oy, sz), (sx, 0, 0), (0, sy, 0)),
                  ((ox, oy, 0), (sx, 0, 0), (0, 0, sz)), ((ox, oy + sy, 0), (sx, 0, 0), (0, 0, sz)),
                  ((ox, oy, 0), (0, sy, 0), (0, 0, sz)), ((ox + sx, oy, 0), (0, sy, 0), (0, 0, sz))]
    o, u, v = (np.array([r[i] for r in rects], np.float64) for i in range(3))
    area = np.linalg.norm(np.cross(u, v), axis=1)
    k = rng.choice(len(rects), size=n, p=area / area.sum())
    a, b = rng.random((n, 1)), rng.random((n, 1))
    pts = o[k] + a * u[k] + b * v[k] + rng.normal(0.0, 0.005, (n, 3))
    return pts.astype(dtype)


def synthetic_head_trajectory(batch: int, seed: int = 0, dtype=np.float64) -> np.ndarray:
    """(batch,4,4) cam_from_world poses of a head-mounted, downward-looking fisheye camera walking a smooth loop in
    synthetic_world_scan's room: head height 1.5-1.8 m, optical axis (camera z) tilted up to ~0.35 rad from straight
    down, heading turning through the walk.  The head stays at least 3 m from every wall, so the network's cuboid
    (x, y in [-s/2, s/2], z in [0, s] in the camera frame) stays within the walls for s <= 2.5; its far face passes
    below the floor, as it does for a standing person.  Rigid: cam_from_world = [R^T | -R^T c] for the camera's
    world orientation R and centre c, computed in fp64 and rounded to `dtype`."""
    rng = np.random.default_rng(seed)
    W, D, _ = ROOM_SIZE
    t = np.arange(batch, dtype=np.float64) / max(batch, 1)
    ph = rng.uniform(0, 2 * np.pi, 5)
    cx = W / 2 + 1.5 * np.sin(2 * np.pi * t + ph[0])
    cy = D / 2 + 0.8 * np.sin(4 * np.pi * t + ph[1])
    cz = 1.65 + 0.15 * np.sin(6 * np.pi * t + ph[2])
    yaw = ph[3] + 2 * np.pi * t
    tilt = 0.2 + 0.15 * np.sin(2 * np.pi * 3 * t + ph[4])
    out = np.zeros((batch, 4, 4), np.float64)
    for i in range(batch):
        zc = np.array([np.sin(tilt[i]) * np.cos(yaw[i]), np.sin(tilt[i]) * np.sin(yaw[i]), -np.cos(tilt[i])])
        xc = np.array([-np.sin(yaw[i]), np.cos(yaw[i]), 0.0])
        yc = np.cross(zc, xc)
        R = np.stack([xc, yc, zc], axis=1)                  # columns: camera axes in world coordinates
        c = np.array([cx[i], cy[i], cz[i]])
        out[i, :3, :3] = R.T
        out[i, :3, 3] = -R.T @ c
        out[i, 3, 3] = 1.0
    return out.astype(dtype)


def stage_state_shapes(with_intersection: bool = False, num_joints: int = 15):
    """(key, shape) of every post-backbone state-dict entry of VoxelNetwork_depth (`process_features.*`,
    `volume_net.*`), derived from the module classes themselves (no GPU, no golden manifest needed)."""
    from ..network.v2v import V2VModel
    m = V2VModel(65 if with_intersection else 33, num_joints)
    shapes = [("process_features.0.weight", (32, 256, 1, 1)), ("process_features.0.bias", (32,))]
    shapes += [("volume_net." + k, tuple(v.shape)) for k, v in m.state_dict().items()]
    return shapes

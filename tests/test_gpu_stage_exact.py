"""The stage's other kernels element by element against float64 references (tests/stage_reference.py): the backbone
hand-off, the 1x1 feature conv (tensor-core split and CUDA-core forms), the unprojection, the soft-argmax and the
output-#2 / generic grid_sample kernels.

Integer fixtures are exact in fp32 at every partial sum (each test asserts that on its data) and must match bit for
bit; Gaussian fixtures must lie within the bounds derived in stage_reference.  Every destination starts as a NaN
(0xFFFF for 16-bit volumes) sentinel and holds one frame more than the launch writes: every element of the launched
frames must be written and the spare frame must stay untouched.  The CPU tests anchor the hand-off fold against the
packer's blob and show that each bound admits the kernel's arithmetic and rejects a dropped term."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests import stage_reference as sr
from tests import util
from tests import v2v_reference as vr
from tests.test_gpu_v2v_exact import check_untouched, decode

F64 = torch.float64
F16_RUN = os.environ.get("SCENEEGO_ACT_DTYPE", "bf16").lower() in ("f16", "fp16", "float16")
MODES = ["exact", "random"]
IMG_H, IMG_W = 1024, 1280


def _nan(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device="cuda")


def _assert_spare(t, B, where):
    assert bool(torch.isnan(t[B:]).all()), f"{where}: the spare frame was written"


def _assert_exact_sums(absum, grid, where):
    """The premise of a bit-exact comparison: every partial sum is a multiple of `grid` below 2^24 grid."""
    a = float(absum.max())
    assert a < 2.0 ** 24 * grid, f"{where}: sum |w| |x| = {a} reaches 2^24 units of {grid}: sums are not exact in fp32"


def _report(where, got, ref):
    print(f"{where}: max |err| / bound = {sr.err_ratio(got, ref):.3e}")


# ---- backbone hand-off ----------------------------------------------------------------------------------------------
def _handoff_modules(mode, seed):
    """ConvTranspose2d(256, 256, 4, 2, 1) + BatchNorm2d + Conv2d(256, 32, 1).  exact: weights k 2^-6 (|k| <= 7), eps = 0,
    var in {1, 4}, gamma in {0.5, 1, 2} (power-of-two scales), beta and mean multiples of 2^-5, 1x1 bias k 2^-6."""
    g = torch.Generator().manual_seed(seed)
    dc = nn.ConvTranspose2d(256, 256, 4, stride=2, padding=1, bias=False)
    bn = nn.BatchNorm2d(256)
    pf = nn.Conv2d(256, 32, 1)
    with torch.no_grad():
        if mode == "exact":
            dc.weight.copy_(torch.randint(-7, 8, dc.weight.shape, generator=g).float() / 64)
            pf.weight.copy_(torch.randint(-7, 8, pf.weight.shape, generator=g).float() / 64)
            pf.bias.copy_(torch.randint(-64, 65, (32,), generator=g).float() / 64)
            vr._set_int_bn(bn, g)
        else:
            dc.weight.copy_(torch.randn(dc.weight.shape, generator=g) * (2.0 / (256 * 4)) ** 0.5)
            pf.weight.copy_(torch.randn(pf.weight.shape, generator=g) * (1.0 / 256) ** 0.5)
            pf.bias.copy_(torch.randn(32, generator=g) * 0.1)
            bn.weight.copy_(torch.rand(256, generator=g) + 0.5)
            bn.bias.copy_(torch.randn(256, generator=g) * 0.1)
            bn.running_mean.copy_(torch.randn(256, generator=g) * 0.1)
            bn.running_var.copy_(torch.rand(256, generator=g) * 1.5 + 0.5)
    return dc.eval(), bn.eval(), pf.eval()


def _handoff_operands(dc, bn, pf):
    w1, shift = sr.handoff_fold(dc.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps)
    w2 = vr.r16(pf.weight.detach().reshape(32, 256).to(F64))
    b2 = pf.bias.detach().to(torch.float32).to(F64)
    return w1, shift, w2, b2


def _handoff_input(mode, B, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    if mode == "exact":
        return torch.randint(-2, 3, (B, 256, h, w), generator=g).to(F64)
    return vr.r16(torch.randn(B, 256, h, w, generator=g).to(F64))


HANDOFF_CASES = [
    # B, h, w: work items of 128 positions (frame = (h + 2) (w + 2) rounded up to 8)
    ("product-1x32x32", 1, 32, 32),           # 10 items
    ("bench-64x32x32", 64, 32, 32),           # 580 items: four rounds of 74 clusters
    ("odd-items-5x16x24", 5, 16, 24),         # 19 items: CTA 1 repeats the last one
    ("single-item-1x1x1", 1, 1, 1),           # 1 item: CTA 1 of the only cluster repeats it and stores nothing
    ("widest-3x1x37", 3, 1, 37),              # halo = HO_GUARD; 3 items
    ("ragged-70x16x16", 70, 16, 16),          # 180 items, the last one partial
]


@pytest.mark.gpu
@pytest.mark.parametrize("multicast", ["1", "0"])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", HANDOFF_CASES, ids=[c[0] for c in HANDOFF_CASES])
def test_handoff(case, mode, multicast, monkeypatch):
    from sceneego_b200 import _lib
    name, B, h, w = case
    monkeypatch.setenv("SCENEEGO_HANDOFF_MULTICAST", multicast)
    dc, bn, pf = _handoff_modules(mode, seed=B + h + w)
    w1, shift, w2, b2 = _handoff_operands(dc, bn, pf)
    x = _handoff_input(mode, B, h, w, seed=B * 7 + h)
    wts, bias = _lib.handoff_pack(dc.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps, pf.weight,
                                  pf.bias, "cuda")
    out = _nan(B + 1, 2 * h, 2 * w, 32)
    _lib.backbone_handoff(x.float().cuda(), wts, bias, out=out[:B])
    torch.cuda.synchronize()
    ref = sr.handoff_ref(x.cuda(), w1, shift, w2, b2)
    where = f"handoff {name} {mode} multicast={multicast}"
    if mode == "exact":
        _assert_exact_sums(ref.A[0], 2.0 ** -8, where + " GEMM 1")
        _assert_exact_sums(ref.A[1], 2.0 ** -14, where + " GEMM 2")
        sr.assert_equal_flat(out[:B], ref.value, where)
    else:
        sr.assert_within_flat(out[:B], ref, where)
        _report(where, out[:B], ref)
    _assert_spare(out, B, where)


@pytest.mark.gpu
def test_handoff_refuses_what_it_cannot_run():
    """w = 38 needs a halo beyond the guard; a batch whose positions reach 2^31 does not fit one launch."""
    from sceneego_b200 import _lib
    dc, bn, pf = _handoff_modules("random", 1)
    wts, bias = _lib.handoff_pack(dc.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps, pf.weight,
                                  pf.bias, "cuda")
    with pytest.raises(_lib.SceneEgoError, match="wider than 38"):
        _lib.backbone_handoff(torch.zeros(1, 256, 2, 38, device="cuda"), wts, bias)
    x = torch.zeros(1, 256, 32, 32, device="cuda")
    ws = torch.zeros(1024, dtype=torch.uint8, device="cuda")
    out = torch.zeros(1, 64, 64, 32, device="cuda")
    frame_cells = (34 * 34 + 7) // 8 * 8
    batch = (2 ** 31 - 4096) // frame_cells + 1           # the arguments are refused before any buffer is touched
    with pytest.raises(_lib.SceneEgoError, match="batch too large"):
        _lib._call("sceneego_backbone_handoff_f32", x, x, batch, 256, 32, 32, wts, bias, ws, out)


# ---- 1x1 feature conv -------------------------------------------------------------------------------------------------
def _fc_operands(kind, B, h, w, seed):
    """kind: 'hh' x and w exact in bf16; 'xl' x = i + j 2^-12 (both bf16 halves nonzero), w exact in bf16; 'wl' x integer,
    w = k 2^-6 + m 2^-16 (both halves nonzero); 'random' Gaussian.  Returns (x, w, b, grid of the partial sums)."""
    g = torch.Generator().manual_seed(seed)
    if kind == "random":
        return (torch.randn(B, 256, h, w, generator=g).to(F64).float().to(F64),
                (torch.randn(32, 256, generator=g) * 0.08).to(F64), (torch.randn(32, generator=g) * 0.1).to(F64), None)
    ints = lambda lo, hi, shape: torch.randint(lo, hi + 1, shape, generator=g).to(F64)
    nonzero = lambda shape: ints(1, 2, shape) * torch.where(ints(0, 1, shape) > 0, 1.0, -1.0)
    b = ints(-64, 64, (32,)) / 64
    if kind == "hh":
        return ints(-2, 2, (B, 256, h, w)), ints(-7, 7, (32, 256)) / 64, b, 2.0 ** -6
    if kind == "xl":
        return nonzero((B, 256, h, w)) + ints(-7, 7, (B, 256, h, w)) / 4096, ints(-7, 7, (32, 256)) / 64, b, 2.0 ** -18
    k = ints(1, 7, (32, 256)) * torch.where(ints(0, 1, (32, 256)) > 0, 1.0, -1.0)
    return ints(-2, 2, (B, 256, h, w)), k / 64 + ints(-3, 3, (32, 256)) / 65536, b, 2.0 ** -16


def _fc_run(x, w, b, misaligned=False):
    from sceneego_b200 import _lib
    B, _, h, wd = x.shape
    wt = w.float().cuda()
    if misaligned:                                         # a weight pointer 4 bytes past a 16-byte boundary
        store = torch.empty(32 * 256 + 1, device="cuda")
        store[1:].copy_(wt.reshape(-1))
        wt = store[1:].view(32, 256)
        assert wt.data_ptr() % 16 == 4
    out = _nan(B + 1, h, wd, 32)
    _lib.feature_conv1x1(x.float().cuda().contiguous(), wt, b.float().cuda(), out=out[:B])
    torch.cuda.synchronize()
    return out


FC_SHAPES = [("bench-64x64x64", 64, 64, 64), ("hw-below-128", 3, 8, 8), ("hw-480", 2, 20, 24),
             ("hw-117-odd", 2, 9, 13), ("hw-405", 2, 15, 27)]
FC_PATHS = ["tensor-core", "simt-env", "simt-misaligned"]


@pytest.mark.gpu
@pytest.mark.parametrize("path", FC_PATHS)
@pytest.mark.parametrize("kind", ["hh", "xl", "wl", "random"])
@pytest.mark.parametrize("shape", FC_SHAPES, ids=[s[0] for s in FC_SHAPES])
def test_feature_conv(shape, kind, path, monkeypatch):
    name, B, h, w = shape
    if path == "simt-env":
        monkeypatch.setenv("SCENEEGO_FEATURE_CONV_SIMT", "1")
    else:
        monkeypatch.delenv("SCENEEGO_FEATURE_CONV_SIMT", raising=False)
    x, wt, b, grid = _fc_operands(kind, B, h, w, seed=B + h * w)
    if kind == "xl":
        xh, xl = sr.bf16_split(x)
        assert torch.equal(xh + xl, x) and float((xl != 0).to(F64).mean()) > 0.8
    if kind == "wl":
        wh, wl = sr.bf16_split(wt)
        assert torch.equal(wh + wl, wt) and float((wl != 0).to(F64).mean()) > 0.8
    out = _fc_run(x, wt, b, misaligned=path == "simt-misaligned")
    ref = sr.feature_conv_ref(x.cuda(), wt, b, tensor_core=path == "tensor-core")
    where = f"feature_conv {name} {kind} {path}"
    if grid is not None:
        _assert_exact_sums(ref.A, grid, where)
        sr.assert_equal_flat(out[:B], ref.value, where)
    else:
        sr.assert_within_flat(out[:B], ref, where)
        _report(where, out[:B], ref)
    _assert_spare(out, B, where)


# ---- unprojection ----------------------------------------------------------------------------------------------------
def _cam():
    from sceneego_b200.utils.fisheye.FishEyeCalibrated import FishEyeCameraCalibrated
    return FishEyeCameraCalibrated(util.CALIB).calib_struct(IMG_W, IMG_H)


def _crafted_coords(rng, n):
    """(ix, iy) targets on the edges the kernel must get right: both sides of 16-px source-cell edges, the pad boundaries
    x = 127 / 128 and 1151 / 1152, the image border."""
    edge_x = 128 + 16 * rng.integers(1, 63, n) + rng.choice([-0.75, -0.5, -0.25, 0.0, 0.25, 0.5], n)
    edge_y = 16 * rng.integers(1, 63, n) + rng.choice([-0.75, -0.5, -0.25, 0.0, 0.25, 0.5], n)
    pads = np.array([126.5, 127.0, 127.25, 127.5, 127.75, 128.0, 128.5, 1150.5, 1151.0, 1151.5, 1151.75, 1152.0,
                     1152.5, 0.0, 0.5, 1278.5, 1279.0])
    ys = np.concatenate([edge_y[: len(pads)], [0.0, 0.5, 1022.5, 1023.0, 511.5]])
    xs = np.concatenate([pads, rng.uniform(128, 1152, 5)])
    return np.concatenate([edge_x, xs]), np.concatenate([edge_y, ys])


def _special_grid_values():
    one = np.float32(1.0)
    vals = [one, -one, np.nextafter(one, np.float32(2)), np.nextafter(-one, np.float32(-2)),
            np.float32(1e30), np.float32(-1e30), np.float32(0.0)]
    return np.array([(a, b) for a in vals for b in vals], np.float32)


def _unproject_grid(V, seed):
    """(V^3, 2) f32 grid: uniform in [-1.1, 1.1]^2 with crafted points planted at random voxels."""
    rng = np.random.default_rng(seed)
    N = V ** 3
    grid = rng.uniform(-1.1, 1.1, (N, 2)).astype(np.float32)
    tx, ty = _crafted_coords(rng, 2000)
    crafted = np.concatenate([np.stack([sr.grid_for(tx, IMG_W), sr.grid_for(ty, IMG_H)], 1), _special_grid_values()])
    where = rng.choice(N, len(crafted), replace=False)
    grid[where] = crafted
    return grid


def _unproject_ref(feat, grid):
    ix, iy = sr.sample_coords(grid[:, 0], IMG_W), sr.sample_coords(grid[:, 1], IMG_H)
    return sr.sample_ref(sr.unproject_gather(feat, IMG_H, IMG_W), sr.bilinear_taps(ix, iy), grid.shape[0])


def _feat(mode, B, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    if mode == "exact":
        return torch.randint(-8, 9, (B, h, w, 32), generator=g).to(F64)
    return torch.randn(B, h, w, 32, generator=g).to(F64)


UNPROJECT_CASES = [
    # id, V, B, source h, w
    ("V64-B1", 64, 1, 64, 64),
    ("V64-B9", 64, 9, 64, 64),                 # two frames per thread, the last group ragged
    ("V64-B64", 64, 64, 64, 64),               # four frames per thread: the bench launch
    ("V128-B1", 128, 1, 64, 64),
    ("V48-B33", 48, 33, 64, 64),               # V not a power of two; four frames per thread, one in the last group
    ("V96-B2", 96, 2, 64, 64),
    ("V64-B2-src20x27", 64, 2, 20, 27),        # the division path of the nearest source cell
]


def _run_unproject(feat, grid, calib, V, B, out_f32=None, out16=None, lay=None, extra=0):
    from sceneego_b200 import _lib
    _lib.unproject(feat.float().cuda().contiguous(), grid, calib, V, 2.0, IMG_H, IMG_W, out_f32, out16, lay,
                   extra_zero_planes=extra)
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", UNPROJECT_CASES, ids=[c[0] for c in UNPROJECT_CASES])
def test_unproject_table_mode(case, mode):
    """Table mode against the float64 sampler, every voxel and channel; the 16-bit planar output equals R16 of the f32
    output in the plain layout (two cleared zero planes behind the features)."""
    from sceneego_b200 import _lib
    name, V, B, h, w = case
    feat = _feat(mode, B, h, w, seed=V + B + h)
    grid = _unproject_grid(V, seed=V * 3 + B)
    out = _nan(B + 1, 32, V, V, V)
    lay = _lib.vol_layout(V, 1, B + 1)
    vol = _lib.alloc_volume(lay, 48, "cuda")
    vol.view(torch.int16).fill_(-1)
    _run_unproject(feat, torch.from_numpy(grid).cuda(), None, V, B, out[:B], vol, lay, extra=2)
    where = f"unproject {name} {mode}"
    _assert_spare(out, B, where)
    fc = feat.cuda()
    for b0 in range(0, B, 8):                              # the float64 reference in slices of 8 frames
        b1 = min(B, b0 + 8)
        ref = _unproject_ref(fc[b0:b1], grid)
        got = out[b0:b1].reshape(b1 - b0, 32, -1).transpose(1, 2)
        sr.assert_within_flat(got, ref, f"{where} frames {b0}..")
        if b0 == 0:
            _report(where, got, ref)
    got16 = decode(vol, lay, B, 48)
    sr.assert_equal_flat(got16[:, :32], vr.r16(out[:B].to(F64)), where + " 16-bit planar output")
    assert not bool(got16[:, 32:].any()), f"{where}: the zero planes behind the features were not cleared"
    check_untouched(vol, lay, B, where + " 16-bit planar output")


@pytest.mark.gpu
@pytest.mark.parametrize("V,B,h,w", [(64, 2, 64, 64), (48, 9, 64, 64), (96, 33, 20, 27)])
def test_unproject_fused_equals_table_mode(V, B, h, w):
    """The fused projection computes the same fp32 grid as sceneego_project_voxels (same project_voxel and
    normalise_px with explicit _rn intrinsics, same lo / step), so its output equals table mode bit for bit, in f32 and
    in all three 16-bit layouts."""
    from sceneego_b200 import _lib
    calib = _cam()
    _, grid = _lib.project_voxels(calib, V, 2.0, (IMG_H, IMG_W), "cuda")
    feat = _feat("random", B, h, w, seed=V + B)
    outs = {}
    for fused in (False, True):
        out = _nan(B + 1, 32, V, V, V)
        _run_unproject(feat, None if fused else grid, calib if fused else None, V, B, out[:B])
        _assert_spare(out, B, f"unproject fused={fused} V{V} B{B}")
        outs[fused] = out
    sr.assert_equal_flat(outs[True][:B], outs[False][:B], f"unproject V{V} B{B}: fused vs table mode")
    want16 = vr.r16(outs[False][:B].to(F64))
    for kind in ("plain", "s2d", "zwin"):
        for fused in (False, True):
            where = f"unproject V{V} B{B} fused={fused} {kind} layout"
            if kind == "plain":
                lay, ch, extra = _lib.vol_layout(V, 1, B + 1), 40, 1
            elif kind == "s2d":
                lay, ch, extra = _lib.vol_layout_s2d(V, B + 1), 33 * 8, 1
            else:
                lay, ch, extra = _lib.vol_layout_zwin(V, B + 1), 40, 1
            vol = _lib.alloc_volume(lay, ch, "cuda")
            vol.view(torch.int16).fill_(-1)
            _run_unproject(feat, None if fused else grid, calib if fused else None, V, B, None, vol, lay, extra)
            got = _lib.unpack_volume(vol, lay, B, 33).to(F64)
            sr.assert_equal_flat(got[:, :32], want16, where)
            assert not bool(got[:, 32].any()), f"{where}: the occupancy plane was not cleared"
            check_untouched(vol, lay, B, where)


# ---- soft-argmax ------------------------------------------------------------------------------------------------------
def _coords(V):
    from oracle import sceneego_oracle as orc
    c = orc.build_coord_volume(V, 2.0)
    axis = torch.stack([c[:, 0, 0, 0], c[0, :, 0, 1], c[0, 0, :, 2]]).contiguous()
    return c.reshape(-1, 3).contiguous(), axis


def _softargmax(x, mult, softmax, mode, V):
    """One launch with sentinel-filled keypoint and volume buffers of one spare frame; returns (kp, vol) buffers."""
    from sceneego_b200 import _lib
    B, J = x.shape[:2]
    coords, axis = _coords(V)
    lib = _lib.load_library()
    ws = torch.empty(lib.sceneego_softargmax_workspace_bytes(B, J, V) // 4, device="cuda")
    kp, vol = _nan(B + 1, J, 3), _nan(B + 1, J, V, V, V)
    _lib._call("sceneego_softargmax3d_f32", x, x, B, J, V, C.c_float(mult), int(softmax),
               axis.cuda() if mode == "axis" else None, coords.cuda() if mode == "coords" else None, kp[:B], vol[:B], ws)
    torch.cuda.synchronize()
    return kp, vol, coords


def _logits(kind, B, J, V, seed):
    g = torch.Generator().manual_seed(seed)
    N = V ** 3
    if kind == "gauss":
        return torch.randn(B, J, N, generator=g) * 3
    if kind == "uniform":
        return torch.full((B, J, N), 0.75)
    if kind == "dominant":
        x = torch.randn(B, J, N, generator=g)
        x[:, :, torch.randint(0, N, (1,), generator=g)] = 60.0
        return x
    if kind == "sparse":                                   # -inf everywhere but a few voxels: whole chunks are -inf
        x = torch.full((B, J, N), float("-inf"))
        for b in range(B):
            for j in range(J):
                idx = torch.randint(0, N, (3,), generator=g)
                x[b, j, idx] = torch.randn(3, generator=g) * 2
        return x
    raise ValueError(kind)


SA_CASES = [
    # id, V, B, J, logits, multiplier, softmax
    ("V4", 4, 2, 3, "gauss", 1.0, True),
    ("V12", 12, 2, 3, "gauss", 1.0, True),
    ("V96", 96, 1, 2, "gauss", 1.0, True),
    ("bench-V64-B64-J15", 64, 64, 15, "gauss", 1.0, True),
    ("V128-B1", 128, 1, 15, "gauss", 1.0, True),
    ("uniform-V64", 64, 1, 2, "uniform", 1.0, True),
    ("uniform-V12", 12, 2, 2, "uniform", 1.0, True),
    ("dominant-V64", 64, 1, 3, "dominant", 1.0, True),
    ("sparse-inf-V64", 64, 1, 3, "sparse", 1.0, True),
    ("sparse-inf-V32", 32, 2, 2, "sparse", 1.0, True),
    ("negative-multiplier", 32, 2, 3, "gauss", -0.5, True),
    ("no-softmax-V32", 32, 2, 3, "gauss", 0.7, False),
    ("no-softmax-V12", 12, 2, 3, "gauss", 1.0, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("coord_mode", ["axis", "coords"])
@pytest.mark.parametrize("case", SA_CASES, ids=[c[0] for c in SA_CASES])
def test_softargmax(case, coord_mode):
    name, V, B, J, kind, mult, softmax = case
    x = _logits(kind, B, J, V, seed=V + B + J).reshape(B, J, V, V, V).cuda()
    kp, vol, coords = _softargmax(x, mult, softmax, coord_mode, V)
    where = f"softargmax {name} {coord_mode}"
    _assert_spare(kp, B, where + " keypoints")
    _assert_spare(vol, B, where + " volume")
    kref, vref = sr.softargmax_ref(x.reshape(B, J, -1).to(F64), mult, softmax, coords.to(F64))
    got_vol = vol[:B].reshape(B, J, -1)
    if softmax:
        sr.assert_within_flat(got_vol, vref, where + " volume")
        _report(where + " volume", got_vol, vref)
    else:
        sr.assert_equal_flat(got_vol, vref.value, where + " volume")
    sr.assert_within_flat(kp[:B], kref, where + " keypoints")
    _report(where + " keypoints", kp[:B], kref)
    if kind == "uniform":
        mean = coords.to(F64).mean(0).cuda()
        assert torch.allclose(kref.value, mean.expand_as(kref.value), rtol=0, atol=1e-12)


# ---- output #2 and the generic grid_sample -------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("h,w,up,pad", [(64, 64, 1024, 128), (32, 40, 1024, 128), (32, 20, 512, 0), (16, 24, 256, 0)])
def test_features_upsample_pad(h, w, up, pad):
    """A pure copy: torch.equal to F.pad(F.interpolate(feat, (up, up)), (pad, pad)) of the same device tensor.  The
    ratios h / up and w / up are dyadic, so torch's fp32 source index floor(dst * (w / up)) is the exact quotient the
    kernel computes."""
    from sceneego_b200 import _lib
    B = 2
    feat = torch.randn(B, h, w, 32, generator=torch.Generator().manual_seed(h + w)).cuda()
    out = _nan(B + 1, 32, up, up + 2 * pad)
    _lib.features_upsample_pad(feat, up, pad, out=out[:B])
    torch.cuda.synchronize()
    want = F.pad(F.interpolate(feat.permute(0, 3, 1, 2), (up, up)), (pad, pad))
    assert torch.equal(out[:B], want), f"upsample_pad {h}x{w} -> {up} pad {pad}"
    _assert_spare(out, B, f"upsample_pad {h}x{w}")


@pytest.mark.gpu
def test_features_upsample_pad_refuses_a_ragged_height():
    from sceneego_b200 import _lib
    with pytest.raises(_lib.SceneEgoError, match="multiple of h"):
        _lib.features_upsample_pad(torch.zeros(1, 24, 32, 32, device="cuda"), 1024, 128)


GS_CASES = [("37x53-shared", 2, 5, 37, 53, True), ("64x80-per-frame", 3, 32, 64, 80, False),
            ("1024x1280-shared", 1, 4, 1024, 1280, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", GS_CASES, ids=[c[0] for c in GS_CASES])
def test_grid_sample(case, mode):
    """sceneego_grid_sample_f32 (bilinear, zeros, align_corners=True) against the float64 sampler, with crafted grid
    values: the image border, +-1 exactly and one ulp outside, +-1e30."""
    from sceneego_b200 import _lib
    name, B, Cc, H, W, shared = case
    g = torch.Generator().manual_seed(H + W)
    rng = np.random.default_rng(H)
    img = (torch.randint(-8, 9, (B, Cc, H, W), generator=g).to(F64) if mode == "exact"
           else torch.randn(B, Cc, H, W, generator=g).to(F64))
    n = 5003
    gb = 1 if shared else B
    grid = rng.uniform(-1.2, 1.2, (gb, n, 2)).astype(np.float32)
    special = _special_grid_values()
    border = np.stack([sr.grid_for(rng.choice([0, 0.5, W - 1.5, W - 1, W - 0.5], 40), W),
                       sr.grid_for(rng.choice([0, 0.5, H - 1.5, H - 1, H - 0.5], 40), H)], 1)
    grid[:, : len(special)] = special
    grid[:, len(special): len(special) + len(border)] = border
    gd = torch.from_numpy(grid).cuda()
    out = _nan(B + 1, Cc, n)
    imf = img.float().cuda()
    _lib._call("sceneego_grid_sample_f32", imf, imf, C.c_void_p(gd.data_ptr()),
               C.c_int64(0 if shared else n * 2), B, Cc, H, W, n, out[:B])
    torch.cuda.synchronize()
    where = f"grid_sample {name} {mode}"
    _assert_spare(out, B, where)
    imc = img.cuda()
    for b in range(B):
        gr = grid[0 if shared else b]
        ix, iy = sr.sample_coords(gr[:, 0], W), sr.sample_coords(gr[:, 1], H)
        ref = sr.sample_ref(sr.image_gather(imc[b:b + 1]), sr.bilinear_taps(ix, iy), n)
        got = out[b:b + 1].transpose(1, 2)
        sr.assert_within_flat(got, ref, f"{where} frame {b}")
        if b == 0:
            _report(where, got, ref)


# ---- both storage builds -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.skipif(F16_RUN, reason="already running on the fp16-storage build")
def test_stage_exact_with_fp16_storage_build():
    """This file's GPU tests on libsceneego_b200_f16.so (one activation dtype per process: a subprocess)."""
    env = dict(os.environ, SCENEEGO_ACT_DTYPE="f16", PYTHONPATH=util.ROOT)
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_stage_exact.py", "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider"], cwd=util.ROOT, env=env, capture_output=True, text=True, timeout=1800)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert " passed" in tail.splitlines()[-1]


# ---- CPU: the hand-off fold equals the packer, and each bound admits the kernel and rejects a dropped term -------------
def _decode_handoff_blob(w_out):
    """The packer's blob as (W1 (cin, cout, 4, 4), W2 (32, 256)) in the storage type: GEMM-1 chunks are
    [parity 4][window half 2][tap 4][K-step 8][k-chunk 2][256 rows][8], the 1x1 weights [K-step 16][k-chunk 2][32][8]."""
    raw = torch.from_numpy(w_out.cpu().numpy().view(np.int16).copy()).view(vr.storage_dtype())
    n1 = 4 * 2 * 4 * 8 * 2 * 256 * 8
    b1 = raw[:n1].view(4, 2, 4, 8, 2, 256, 8)
    tap_k = {(0, 0): 1, (0, 1): 3, (1, 0): 0, (1, 1): 2}        # ho_tap_k(parity bit, t)
    w1 = torch.zeros(256, 256, 4, 4, dtype=vr.storage_dtype())
    for par in range(4):
        for t in range(4):
            ky, kx = tap_k[(par >> 1, t >> 1)], tap_k[(par & 1, t & 1)]
            blk = b1[par, :, t]                                        # (hf, kh, c, co, e): ci = (hf 8 + kh) 16 + c 8 + e
            w1[:, :, ky, kx] = blk.permute(0, 1, 2, 4, 3).reshape(256, 256)
    w2 = raw[n1:].view(16, 2, 32, 8).permute(2, 0, 1, 3).reshape(32, 256)
    return w1, w2


@pytest.mark.parametrize("mode", MODES)
def test_handoff_fold_equals_packer(mode):
    """sceneego_handoff_pack decoded: GEMM-1 weights, 1x1 weights, BN shift and 1x1 bias equal stage_reference's fold
    bit for bit (a weight beyond the fp16 range saturates to 65504 on the fp16 build)."""
    from sceneego_b200 import _lib
    dc, bn, pf = _handoff_modules(mode, seed=3)
    if mode == "random":
        with torch.no_grad():
            dc.weight.view(-1)[5] = 1.0e6
            pf.weight.view(-1)[7] = -3.0e5
    w_out, b_out = _lib.handoff_pack(dc.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps, pf.weight,
                                     pf.bias, "cpu")
    w1, shift, w2, b2 = _handoff_operands(dc, bn, pf)
    got1, got2 = _decode_handoff_blob(w_out)
    assert torch.equal(got1.view(torch.int16), w1.to(vr.storage_dtype()).view(torch.int16))
    assert torch.equal(got2.view(torch.int16), w2.to(vr.storage_dtype()).view(torch.int16))
    assert torch.equal(b_out[:256].to(F64), shift)
    assert torch.equal(b_out[256:].to(F64), b2)


@pytest.mark.skipif(F16_RUN, reason="already running on the fp16-storage build")
def test_handoff_fold_equals_packer_on_fp16_build():
    env = dict(os.environ, SCENEEGO_ACT_DTYPE="f16", PYTHONPATH=util.ROOT)
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_stage_exact.py", "-q", "-x", "-p",
                        "no:cacheprovider", "-k", "fold or bound"], cwd=util.ROOT, env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-1500:]


def _handoff_bound_case():
    dc, bn, pf = _handoff_modules("random", seed=11)
    w1, shift, w2, b2 = _handoff_operands(dc, bn, pf)
    x = _handoff_input("random", 2, 6, 7, seed=12)
    return x, w1, shift, w2, b2, sr.handoff_ref(x, w1, shift, w2, b2)


def test_handoff_bound_admits_the_kernel_arithmetic():
    """fp32 GEMMs in shuffled orders with the R16 hidden layer stay within the propagated bound."""
    x, w1, shift, w2, b2, ref = _handoff_bound_case()
    for seed in range(3):
        got = sr.simulate_handoff(x, w1, shift, w2, b2, seed=seed)
        sr.assert_within_flat(got, ref, f"hand-off model, order {seed}")


def test_handoff_bound_rejects_a_dropped_tap():
    """Deconv tap (ky, kx) = (1, 2) of input channel 9 feeds the outputs of parity (even rows, odd columns).  The
    bound's slack is mostly the 16-bit rounding of the 256 hidden activations, so the tap is dropped from a channel
    eight times as strong as the others (the backbone's ReLU maps have such channels)."""
    x, w1, shift, w2, b2, _ = _handoff_bound_case()
    x[:, 9] *= 8
    ref = sr.handoff_ref(x, w1, shift, w2, b2)
    sr.assert_within_flat(sr.simulate_handoff(x, w1, shift, w2, b2), ref, "hand-off model, strong channel")
    got = sr.simulate_handoff(x, w1, shift, w2, b2, drop=(9, 1, 2))
    bad = ~vr.within_mask(got, ref)
    assert not bool(bad[:, 1::2].any()) and not bool(bad[:, :, 0::2].any()), "the dropped tap reaches other parities"
    frac = float(bad[:, 0::2, 1::2].to(F64).mean())
    assert frac >= 0.10, f"dropping one deconv tap of one channel fails only {frac:.3f} of the elements it feeds"


def _fc_bound_case():
    x, w, b, _ = _fc_operands("random", 2, 9, 13, seed=5)
    return x, w, b, sr.feature_conv_ref(x, w, b)


def test_feature_conv_bound_admits_the_split_mmas():
    x, w, b, ref = _fc_bound_case()
    for seed in range(4):
        got = sr.simulate_feature_conv_tc(x, w, b, seed=seed)
        sr.assert_within_flat(got, ref, f"split-MMA model, order {seed}")


def test_feature_conv_bound_rejects_a_dropped_mma():
    x, w, b, ref = _fc_bound_case()
    got = sr.simulate_feature_conv_tc(x, w, b, drop_xl_wh=True)
    frac = float((~vr.within_mask(got, ref)).to(F64).mean())
    assert frac >= 0.10, f"dropping the xl.wh MMA fails only {frac:.3f} of the elements"


def _sample_bound_case():
    feat = _feat("random", 2, 20, 27, seed=4)
    rng = np.random.default_rng(6)
    gx, gy = rng.uniform(-1.1, 1.1, 6000).astype(np.float32), rng.uniform(-1.1, 1.1, 6000).astype(np.float32)
    tx, ty = _crafted_coords(rng, 500)
    gx = np.concatenate([gx, sr.grid_for(tx, IMG_W)])
    gy = np.concatenate([gy, sr.grid_for(ty, IMG_H)])
    ix, iy = sr.sample_coords(gx, IMG_W), sr.sample_coords(gy, IMG_H)
    gather = sr.unproject_gather(feat, IMG_H, IMG_W)
    return gather, ix, iy, sr.sample_ref(gather, sr.bilinear_taps(ix, iy), len(ix))


def test_sample_bound_admits_merged_taps():
    gather, ix, iy, ref = _sample_bound_case()
    for order in ((0, 1, 2, 3), (3, 2, 1, 0), (1, 3, 0, 2)):
        sr.assert_within_flat(sr.simulate_sample_f32(gather, ix, iy, order), ref, f"merged-tap model, order {order}")


def test_sample_bound_rejects_a_dropped_tap():
    gather, ix, iy, ref = _sample_bound_case()
    got = sr.simulate_sample_f32(gather, ix, iy, drop_tap=1)
    frac = float((~vr.within_mask(got, ref)).to(F64).mean())
    assert frac >= 0.10, f"dropping one bilinear tap fails only {frac:.3f} of the elements"

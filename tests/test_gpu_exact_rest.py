"""The remaining hand-written kernels element by element against float64 references: the pose errors (csrc/eval.cu,
tests/eval_reference.py), the fisheye projection (project_voxels_kernel, world2camera_kernel, tests/stage_reference.py),
the with_intersection product (intersect_kernel) and the volume layout conversions (pack_volume_kernel,
unpack_volume_kernel, occ_expand_zwin_kernel) against an index model written from include/sceneego_b200.h and
csrc/common.cuh, independent of pack_volume / unpack_volume.

Every destination starts as a NaN sentinel (0xFFFF for 16-bit volumes) and holds one frame or row more than the launch
writes: the launched part must be written in full and the spare part must stay untouched.  Layout and intersection
results must match bit for bit in both storage builds; the fp16 build runs in a subprocess.  The CPU tests show that
each bound admits a model of the kernel's arithmetic and rejects a planted defect, and check the index model against
the library's layout maker."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests import eval_reference as er
from tests import stage_reference as sr
from tests import util

F16_RUN = os.environ.get("SCENEEGO_ACT_DTYPE", "bf16").lower() in ("f16", "fp16", "float16")
IMG_H, IMG_W = 1024, 1280
# Output sentinels: quiet NaNs with a payload no kernel produces (a NaN a kernel computes is the canonical one), so an
# element counts as untouched only if its bits are unchanged.
SENTINEL_BITS = {torch.float64: 0x7FF80000DEADBEEF, torch.float32: 0x7FC0BEEF}
_INT = {torch.float64: torch.int64, torch.float32: torch.int32}


def _sentinel(*shape, dtype=torch.float32):
    return torch.full(shape, SENTINEL_BITS[dtype], dtype=_INT[dtype], device="cuda").view(dtype)


def _untouched(t):
    """True when every element of t still holds the sentinel bit pattern."""
    return bool((t.view(_INT[t.dtype]) == SENTINEL_BITS[t.dtype]).all())


def _calib():
    from oracle import sceneego_oracle as orc
    return orc.load_calibration(util.CALIB)


def _cam():
    from sceneego_b200.utils.fisheye.FishEyeCalibrated import FishEyeCameraCalibrated
    return FishEyeCameraCalibrated(util.CALIB).calib_struct(IMG_W, IMG_H)


# ==== pose errors ======================================================================================================
POSE_KINDS = ["generic", "reflected", "planar", "near-planar-1e-4", "near-planar-1e-8", "near-planar-1e-13",
              "near-planar-1e-14", "near-planar-1e-15", "collinear-gt", "collinear-pred", "pred-constant", "gt-constant",
              "equal", "translated"]
POSE_CASES = ([(k, 129, 15) for k in POSE_KINDS] + [("isotropic", 4, 6)]
              + [("generic", B, 15) for B in (1, 127, 128, 100000)] + [("generic", 64, 3), ("generic", 64, 64)])


def _pose_run(pred, gt, scale, outputs=("mpjpe", "pampjpe", "aligned", "gt_out", "transform")):
    """sceneego_pose_errors_f64 on B frames with sentinel-filled outputs of B + 1 frames; returns the outputs (numpy),
    None for the ones passed as NULL."""
    from sceneego_b200 import _lib
    B, J = pred.shape[:2]
    nan = lambda *s: _sentinel(*s, dtype=torch.float64)
    bufs = {"mpjpe": nan(B + 1), "pampjpe": nan(B + 1), "aligned": nan(B + 1, J, 3), "gt_out": nan(B + 1, J, 3),
            "transform": nan(B + 1, 13)}
    p = pred.contiguous().cuda()
    g = gt.contiguous().cuda()
    args = [bufs[k][:B] if k in outputs else None for k in ("mpjpe", "pampjpe", "aligned", "gt_out", "transform")]
    _lib._call("sceneego_pose_errors_f64", p, p, int(p.dtype == torch.float64), g, B, J, int(scale), *args)
    torch.cuda.synchronize()
    out = {}
    for k, t in bufs.items():
        t = t.cpu()
        assert _untouched(t[B:]), f"pose_errors: the spare frame of {k} was written"
        if k in outputs:
            out[k] = t[:B].numpy()
        else:
            assert _untouched(t), f"pose_errors: {k} was written though passed as NULL"
    return out


def _pose_inputs(kind, B, J, dtype, seed):
    pred, gt = er.make_case(kind, B, J, seed)
    pred_t = torch.from_numpy(pred).to(dtype)
    return pred_t, torch.from_numpy(gt), pred_t.to(torch.float64).numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [True, False], ids=["scale", "no-scale"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("case", POSE_CASES, ids=[f"{k}-B{B}-J{J}" for k, B, J in POSE_CASES])
def test_pose_errors(case, dtype, scale):
    kind, B, J = case
    pred_t, gt_t, pred64 = _pose_inputs(kind, B, J, dtype, seed=B + J + len(kind))
    out = _pose_run(pred_t, gt_t, scale)
    ref = er.oracle(pred64, gt_t.numpy(), scale)
    bnd = er.bounds(ref)
    where = f"pose_errors {kind} B{B} J{J} {dtype} scale={scale}"
    errs = er.check(out, ref, bnd, where)
    print(f"{where}: free rotation in {int(bnd['free'].sum())} of {B} frames; max |err| / bound "
          + ", ".join(f"{k} {v:.2e}" for k, v in sorted(errs.items())))
    if kind == "pred-constant":                     # varp = 0: the oracle's c is 1/0 * 0; the kernel agrees on NaN
        assert np.isnan(out["transform"][:, 0]).all() and np.isnan(out["pampjpe"]).all()
        assert np.isnan(ref["c"]).all()
    if kind in ("collinear-gt", "collinear-pred", "gt-constant"):
        assert bnd["free"].all(), f"{where}: the case is meant to have rank C <= 1"
    if kind.startswith("near-planar") or kind == "planar":
        assert not bnd["free"].any(), f"{where}: a near-planar pose has a unique rotation"


@pytest.mark.gpu
def test_pose_errors_nan_frame_stays_in_its_frame():
    pred_t, gt_t, pred64 = _pose_inputs("generic", 129, 15, torch.float32, seed=3)
    pred_t[77, 4, 1] = float("nan")
    out = _pose_run(pred_t, gt_t, True)
    assert np.isnan(out["mpjpe"][77]) and np.isnan(out["pampjpe"][77])
    keep = np.ones(129, bool)
    keep[77] = False
    p64 = pred64.copy()
    p64[77] = gt_t.numpy()[77]                      # any finite frame: it is excluded from the comparison
    ref = er.oracle(p64, gt_t.numpy(), True)
    er.check(out, ref, er.bounds(ref), "pose_errors NaN in frame 77", frames=keep)


@pytest.mark.gpu
@pytest.mark.parametrize("outputs", [("mpjpe", "pampjpe"), ("aligned", "gt_out", "transform"), ("pampjpe",),
                                     ("transform",)])
def test_pose_errors_null_outputs(outputs):
    """Outputs passed as NULL are skipped; the others equal a call with all five outputs bit for bit."""
    pred_t, gt_t, _ = _pose_inputs("generic", 130, 15, torch.float32, seed=9)
    full = _pose_run(pred_t, gt_t, True)
    part = _pose_run(pred_t, gt_t, True, outputs)
    for k in outputs:
        assert np.array_equal(part[k], full[k]), k


def test_pose_reference_is_the_oracle():
    """The batched restatement equals oracle.umeyama / align_skeleton frame by frame."""
    from oracle import sceneego_oracle as orc
    for scale in (True, False):
        pred, gt = er.make_case("generic", 5, 15, seed=1)
        ref = er.oracle(pred, gt, scale)
        al, g = orc.align_skeleton(pred, gt, scale=scale)
        assert np.allclose(ref["aligned"], al, rtol=0, atol=1e-14) and np.allclose(ref["gt_out"], g, rtol=0, atol=1e-15)
        for b in range(5):
            c, R, t = orc.umeyama(ref["P"][b], ref["gt_out"][b])
            assert abs(c - ref["c"][b]) <= 1e-14 and np.abs(R - ref["R"][b]).max() <= 1e-14
            assert np.abs(t - ref["t"][b]).max() <= 1e-14


MODEL_KINDS = ["generic", "reflected", "planar", "near-planar-1e-8", "near-planar-1e-13", "collinear-gt",
               "collinear-pred", "pred-constant", "gt-constant", "translated"]


@pytest.mark.parametrize("scale", [True, False], ids=["scale", "no-scale"])
@pytest.mark.parametrize("kind", MODEL_KINDS)
def test_pose_bound_admits_the_kernel_model(kind, scale):
    """The float64 model of the kernel, summing the joints in the other order, lies within every bound."""
    pred, gt = er.make_case(kind, 10, 15, seed=5)
    pred = pred.astype(np.float32).astype(np.float64)
    ref = er.oracle(pred, gt, scale)
    er.check(er.model(pred, gt, scale, reverse=True), ref, er.bounds(ref), f"model {kind}")


def test_pose_bound_rejects_a_flipped_third_column():
    pred, gt = er.make_case("generic", 10, 15, seed=6)
    ref = er.oracle(pred, gt, True)
    with pytest.raises(AssertionError, match="R:"):
        er.check(er.model(pred, gt, True, flip_r2=True), ref, er.bounds(ref), "flipped R[:, 2]")


@pytest.mark.parametrize("kind", ["near-planar-1e-13", "collinear-gt", "gt-constant"])
def test_pose_checks_reject_the_earlier_v_construction(kind):
    """V[:, c] = C W[c]^T / S[c] with e_c for S[c] <= tiny (the construction before the orthonormal completion):
    a non-orthogonal R on near-planar and rank <= 1 frames."""
    pred, gt = er.make_case(kind, 10, 15, seed=7)
    ref = er.oracle(pred, gt, True)
    with pytest.raises(AssertionError):
        er.check(er.model(pred, gt, True, legacy_v=True), ref, er.bounds(ref), f"earlier V {kind}")


# ==== fisheye projection ===============================================================================================
def _voxel_points(V, side):
    """The kernel's fp32 voxel centres fl(lo + fl(step i)), x-major like project_voxels' index n."""
    step, lo = np.float32(side / (V - 1)), np.float32(-side / 2)
    i = np.arange(V, dtype=np.float32)
    ax, az = lo + step * i, np.float32(0) + step * i
    return np.stack(np.meshgrid(ax, ax, az, indexing="ij"), -1).reshape(-1, 3).astype(np.float32)


def _crafted_points():
    """Regular crafted points: near the optical axis (one voxel step, 1e-3 steps, 1e-20; theta close to +-pi/2),
    X^2 + Y^2 subnormal, behind the camera (z < 0 after the flip), on the horizon (theta close to 0), large but finite
    coordinates."""
    step = np.float32(2.0 / 63)
    pts = []
    for d in (step, step * np.float32(1e-3), np.float32(1e-20), np.float32(3e-20)):
        for Z in (0.5, -0.5, 1.5, 1e-3, -1e-3):
            pts += [(d, 0, Z), (0, d, Z), (-d, d, Z), (d, -d * np.float32(0.5), Z)]
    for Z in (1e-6, -1e-6, 1e-30, -1e-30, 0.0):             # on the horizon: theta -> 0 (and exactly 0)
        pts += [(0.7, 0.2, Z), (-0.3, 0.9, Z)]
    pts += [(1e-20, 1e-20, 1e-8), (5e-20, -2e-20, -3e-9)]
    pts += [(1e18, 2e18, 3e18), (-4e18, 1e17, -1e18), (1e-3, 2e-3, 1e6), (3.0, -4.0, -2.0)]
    return np.array(pts, np.float32)


def _w2c_run(pts):
    from sceneego_b200 import _lib
    n = pts.shape[0]
    out = _sentinel(n + 1, 2)
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    p = torch.from_numpy(pts).cuda()
    _lib._call("sceneego_world2camera_f32", p, C.byref(_cam()), p, n, out[:n], status)
    torch.cuda.synchronize()
    out = out.cpu()
    assert _untouched(out[n:]), "world2camera: the spare row was written"
    o = out.numpy().astype(np.float64)
    return o[:n], int(status.item())


def _check_w2c(got, pts, where):
    ref, rad, _, r2 = sr.project_ref(pts, _calib())
    ok = sr.w2c_within(got, ref, rad)
    if not ok.all():
        i = np.argwhere(~ok)[0]
        raise AssertionError(f"{where}: {(~ok).sum()} of {ok.size} outside the bound; point {pts[i[0]]}: got "
                             f"{got[tuple(i)]!r}, want {ref[tuple(i)]!r} +- {rad[tuple(i)]:.3e}")
    return float((np.abs(got - ref) / rad).max())


@pytest.mark.gpu
@pytest.mark.parametrize("side", [2.0, 3.0, 1.7])
@pytest.mark.parametrize("V", [48, 64, 96, 128])
def test_project_voxels(V, side):
    """px and the normalised grid of every voxel centre against the float64 expression; status stays 0 (no voxel
    centre of an even V lies on the optical axis, which the test asserts)."""
    from sceneego_b200 import _lib
    N = V ** 3
    px = _sentinel(N + 1, 2)
    grid = _sentinel(N + 1, 2)
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    _lib._call("sceneego_project_voxels_f32", px, C.byref(_cam()), V, C.c_float(side), IMG_H, IMG_W, px[:N], grid[:N],
               status)
    torch.cuda.synchronize()
    px, grid = px.cpu(), grid.cpu()
    assert _untouched(px[N:]) and _untouched(grid[N:]), "project_voxels: the spare row was written"
    px, grid = px.numpy().astype(np.float64), grid.numpy().astype(np.float64)
    pts = _voxel_points(V, side)
    ref, rad, _, r2 = sr.project_ref(pts, _calib())
    assert (r2 > 0).all() and int(status.item()) == 0
    where = f"project_voxels V{V} side {side}"
    ratio = _check_w2c(px[:N], pts, where + " px")
    gref, grad = sr.normalise_ref(ref, rad, IMG_H, IMG_W)
    ok = sr.w2c_within(grid[:N], gref, grad)
    assert ok.all(), f"{where} grid: {(~ok).sum()} elements outside the bound"
    print(f"{where}: max |err| / bound px {ratio:.3e}, grid {float((np.abs(grid[:N] - gref) / grad).max()):.3e}")


@pytest.mark.gpu
def test_world2camera_crafted_points():
    pts = np.concatenate([_crafted_points(), _voxel_points(48, 1.7)[::37]])
    got, status = _w2c_run(pts)
    assert status == 0
    print(f"world2camera crafted: max |err| / bound {_check_w2c(got, pts, 'world2camera crafted'):.3e}")
    # the fp32 oracle lies in the same bound
    from oracle import sceneego_oracle as orc
    _check_w2c(orc.world2camera_f32(_calib(), torch.from_numpy(pts)).double().numpy(), pts, "oracle crafted")


@pytest.mark.gpu
def test_world2camera_degenerate_points():
    """r = 0 exactly (on the axis, or X^2 + Y^2 underflowing in fp32): px = the centre and the status flag, set exactly
    when some r == 0.  torch.norm in the oracle does not rescale either: it gives 0 for X = Y = 1e-23 and raises 'norm
    is zero!' like the kernel's binding.  X^2 overflowing: r = inf, so theta = 0 and X / r = 0; kernel and oracle both
    return the centre, where the exact expression would not.  NaN coordinates give NaN and leave the flag alone."""
    from oracle import sceneego_oracle as orc
    from sceneego_b200 import _lib
    a, cx, cy = sr.w2c_coeffs(_calib())
    regular = _crafted_points()[:8]
    for bad in ([0, 0, 0.5], [1e-23, -1e-23, 0.5], [0, 3e-39, -0.2]):
        pts = np.concatenate([regular, np.array([bad], np.float32)])
        got, status = _w2c_run(pts)
        assert status == 1, bad
        assert got[-1, 0] == cx and got[-1, 1] == cy
        _check_w2c(got[:-1], pts[:-1], f"world2camera beside {bad}")
        with pytest.raises(Exception, match="norm is zero"):
            orc.world2camera_f32(_calib(), torch.from_numpy(pts))
        with pytest.raises(Exception, match="norm is zero"):
            _lib.world2camera(_cam(), torch.from_numpy(pts).cuda())
    special = np.array([[1e20, 0.5, 1.0], [-3e19, 2e19, -1.0], [np.nan, 0.2, 1.0], [0.3, 0.2, np.nan]], np.float32)
    pts = np.concatenate([regular, special])
    got, status = _w2c_run(pts)
    assert status == 0
    want = orc.world2camera_f32(_calib(), torch.from_numpy(pts)).double().numpy()
    assert got[8, 0] == cx and got[8, 1] == cy and got[9, 0] == cx and got[9, 1] == cy
    assert np.array_equal(got[8:10], want[8:10])
    assert np.isnan(got[10:]).all()


def _bound_points():
    return np.concatenate([_voxel_points(64, 2.0)[::5], _crafted_points()])


def test_projection_bound_admits_fp32_models():
    """The fp32 oracle and a NumPy float32 model whose atan is off by up to the full ulp budget lie in the bound."""
    from oracle import sceneego_oracle as orc
    pts = _bound_points()
    _check_w2c(orc.world2camera_f32(_calib(), torch.from_numpy(pts)).double().numpy(), pts, "oracle")
    for seed in range(3):
        _check_w2c(sr.simulate_project_f32(pts, _calib(), atan_ulps=sr.ATANF_ULP, seed=seed), pts, f"model {seed}")


@pytest.mark.parametrize("defect", ["drop-a10", "swap-centre", "no-flip"])
def test_projection_bound_rejects_a_planted_defect(defect):
    """a10 is the smallest term of the W2C polynomial, yet a10 theta^10 reaches 2.4 px at the volume's widest angle
    (theta = -1.56); dropping it must fail most voxels."""
    pts = _voxel_points(64, 2.0)
    kw = {"drop-a10": dict(drop=10), "swap-centre": dict(swap_centre=True), "no-flip": dict(no_flip=True)}[defect]
    got = sr.simulate_project_f32(pts, _calib(), **kw)
    ref, rad, _, _ = sr.project_ref(pts, _calib())
    frac = float((~sr.w2c_within(got, ref, rad)).mean())
    assert frac >= 0.5, f"{defect} fails only {frac:.3f} of the voxels"


# ==== volume layouts: an index model from include/sceneego_b200.h and csrc/common.cuh =================================
class Lay:
    """The layout maker's formulas (sceneego_vol_layout_make, _s2d, _zwin)."""

    def __init__(self, side, pad, batch, s2d=0, zwin=0):
        self.side, self.pad, self.s2d, self.zwin = side, pad, s2d, zwin
        self.pitch_y = side + pad
        self.pitch_x = self.pitch_y ** 2
        g = pad * (self.pitch_x + self.pitch_y + 1)
        self.guard = (g + 7) // 8 * 8
        self.frame_pitch = (self.guard + side * self.pitch_x + 7) // 8 * 8
        self.plane_stride = batch * self.frame_pitch + self.guard + 1024 + 8


def model_layout(kind, S, batch):
    """kind: plain (pad 1), pad3 (the 65-channel input), s2d (full side S), zwin."""
    if kind == "s2d":
        return Lay(S // 2, 2, batch, s2d=1)
    return Lay(S, {"plain": 1, "pad3": 3, "zwin": 3}[kind], batch, zwin=int(kind == "zwin"))


def vol_pos(L, b, x, y, z):
    return b * L.frame_pitch + L.guard + x * L.pitch_x + y * L.pitch_y + z


def elem_index(L, b, x, y, z, ch):
    """16-bit element of channel ch of voxel (x, y, z) (full-resolution coordinates); the z-window occupancy: the
    voxel's own entry (3) of its cell.  Tensors of int64."""
    if L.zwin and ch >= 32:
        return (4 * L.plane_stride + vol_pos(L, b, x, y, z)) * 8 + 3
    if L.s2d:
        par = ((x & 1) << 2) | ((y & 1) << 1) | (z & 1)
        pos = vol_pos(L, b, x >> 1, y >> 1, z >> 1)
        if ch < 32:
            return ((par * 4 + ch // 8) * L.plane_stride + pos) * 8 + ch % 8
        return (32 * L.plane_stride + pos) * 8 + par
    return ((ch // 8) * L.plane_stride + vol_pos(L, b, x, y, z)) * 8 + ch % 8


def _grid(B, S):
    b, x, y, z = torch.meshgrid(torch.arange(B), torch.arange(S), torch.arange(S), torch.arange(S), indexing="ij")
    return b, x, y, z


def storage_bits(x, f16):
    """Round-to-nearest-even into the storage type, as int16 bits.  fp16: cvt.rn.satfinite sends +-inf and values
    beyond the range to +-65504 (torch's .to(float16) would give inf)."""
    x = x.to(torch.float32)
    if f16:
        x = torch.where(torch.isnan(x), x, x.clamp(-65504.0, 65504.0))
        return x.to(torch.float16).view(torch.int16)
    return x.to(torch.bfloat16).view(torch.int16)


def decode_bits(bits, f16):
    return bits.view(torch.float16 if f16 else torch.bfloat16).to(torch.float32)


def pack_expect(buf_bits, x, L, c_offset, f16):
    """Expected buffer after pack_volume(x, c_offset) over `buf_bits` (flat int16)."""
    out = buf_bits.clone()
    B, c, S = x.shape[0], x.shape[1], x.shape[2]
    b, X, Y, Z = _grid(B, S)
    bits = storage_bits(x, f16)
    for ch in range(c):
        oc = ch + c_offset
        if L.zwin and oc >= 32:
            if oc == 32:                                  # the cell occ[x][y][z-3 .. z+4], zeros beyond the volume
                base = (4 * L.plane_stride + vol_pos(L, b, X, Y, Z)) * 8
                for e in range(8):
                    zz = Z + e - 3
                    inside = (zz >= 0) & (zz < S)
                    v = bits[b, ch, X, Y, zz.clamp(0, S - 1)]
                    out[(base + e).reshape(-1)] = torch.where(inside, v, torch.zeros_like(v)).reshape(-1)
            continue
        if L.s2d and oc > 32:
            continue
        out[elem_index(L, b, X, Y, Z, oc).reshape(-1)] = bits[:, ch].reshape(-1)
    return out


def _pack_input(B, c, S, seed, f16):
    """Gaussian values with planted specials: +-0, +-inf, values beyond fp16's range, storage subnormals, ties."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, c, S, S, S, generator=g) * 3
    sub = 2.0 ** -20 if f16 else 2.0 ** -130
    specials = torch.tensor([0.0, -0.0, float("inf"), float("-inf"), 7e4, -1e5, 65519.0, 65520.0, sub, -3 * sub,
                             1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, 1.0 + 2.0 ** -11, 3.4e38])
    idx = torch.randint(0, x.numel(), (specials.numel() * 40,), generator=g)
    x.view(-1)[idx] = specials.repeat(40)
    return x


LAYOUT_CASES = [("plain", 16, 2, 24, 0), ("plain", 12, 3, 16, 8), ("pad3", 16, 2, 40, 8), ("s2d", 16, 2, 33, 0),
                ("s2d", 12, 1, 9, 24), ("zwin", 16, 2, 33, 0), ("zwin", 12, 2, 1, 32), ("zwin", 10, 1, 5, 28)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", LAYOUT_CASES, ids=[f"{k}-S{S}-B{B}-c{c}-off{o}" for k, S, B, c, o in LAYOUT_CASES])
def test_pack_volume(case):
    """Every written element equals the storage rounding of its input and nothing else changes."""
    from sceneego_b200 import _lib
    kind, S, B, c, off = case
    f16 = _lib.act_dtype_name() == "f16"
    L = model_layout(kind, S, B + 1)
    lay = (_lib.vol_layout_s2d(S, B + 1) if kind == "s2d" else _lib.vol_layout_zwin(S, B + 1) if kind == "zwin"
           else _lib.vol_layout(S, L.pad, B + 1))
    assert lay.plane_stride == L.plane_stride and lay.guard == L.guard and lay.frame_pitch == L.frame_pitch
    planes = 33 if kind == "s2d" else 5 if kind == "zwin" else (off + c + 7) // 8
    buf = _lib.alloc_volume(lay, planes * 8, "cuda")
    buf.view(torch.int16).fill_(-1)
    before = buf.view(torch.int16).reshape(-1).cpu()
    x = _pack_input(B, c, S, seed=S + c + off, f16=f16)
    _lib.pack_volume(x.cuda(), buf, lay, c_offset=off)
    torch.cuda.synchronize()
    got = buf.view(torch.int16).reshape(-1).cpu()
    want = pack_expect(before, x, L, off, f16)
    bad = got != want
    assert not bool(bad.any()), (f"pack {case}: {int(bad.sum())} elements differ, first at "
                                 f"{bad.nonzero()[:6, 0].tolist()}")


@pytest.mark.gpu
@pytest.mark.parametrize("case", LAYOUT_CASES, ids=[f"{k}-S{S}-B{B}-c{c}-off{o}" for k, S, B, c, o in LAYOUT_CASES])
def test_unpack_volume(case):
    """A buffer of random bit patterns read through the index model; NaN patterns must read as NaN."""
    from sceneego_b200 import _lib
    kind, S, B, c, off = case
    c = min(off + c, 33) if kind in ("s2d", "zwin") else off + c
    f16 = _lib.act_dtype_name() == "f16"
    L = model_layout(kind, S, B + 1)
    lay = (_lib.vol_layout_s2d(S, B + 1) if kind == "s2d" else _lib.vol_layout_zwin(S, B + 1) if kind == "zwin"
           else _lib.vol_layout(S, L.pad, B + 1))
    planes = 33 if kind == "s2d" else 5 if kind == "zwin" else (c + 7) // 8
    g = torch.Generator().manual_seed(S * 7 + c)
    bits = torch.randint(-32768, 32768, (planes * 8 * L.plane_stride,), generator=g, dtype=torch.int32).to(torch.int16)
    buf = bits.cuda().view(_lib.act_torch_dtype()).view(planes, L.plane_stride, 8)
    out = _sentinel(B + 1, c, S, S, S)
    _lib._call("sceneego_unpack_volume_f32", buf, buf, C.byref(lay), B, c, out[:B])
    torch.cuda.synchronize()
    out = out.cpu()
    assert _untouched(out[B:]), "unpack: the spare frame was written"
    b, X, Y, Z = _grid(B, S)
    vals = decode_bits(bits, f16)
    for ch in range(c):
        want = vals[elem_index(L, b, X, Y, Z, ch)]
        got = out[:B, ch]
        same = (got == want) | (torch.isnan(got) & torch.isnan(want))
        same &= (torch.signbit(got) == torch.signbit(want)) | torch.isnan(want)
        assert bool(same.all()), f"unpack {case} channel {ch}: {int((~same).sum())} elements differ"


@pytest.mark.gpu
@pytest.mark.parametrize("V,B", [(48, 3), (64, 2), (96, 2), (8, 5)])
def test_occ_expand_zwin(V, B):
    """Every real cell of the occupancy plane = occ[x][y][z-3 .. z+4] (zeros beyond the volume), stale cells
    overwritten, pad / guard cells and the spare frame untouched, the grid left all-zero."""
    from sceneego_b200 import _lib
    f16 = _lib.act_dtype_name() == "f16"
    lay = _lib.vol_layout_zwin(V, B + 1)
    L = model_layout("zwin", V, B + 1)
    g = torch.Generator().manual_seed(V + B)
    occ = (torch.rand(B, V, V, V, generator=g) < 0.3).float()
    occ[:, :, :, :3] = 1.0                               # the z < 3 and z > V - 5 edges are occupied
    occ[:, :, :, V - 4:] = 1.0
    occ[0, 1] = 0.0                                      # an empty row plane
    buf = _lib.alloc_volume(lay, 40, "cuda")
    flat = buf.view(torch.int16).reshape(-1)
    flat.fill_(-1)
    b, X, Y, Z = _grid(B, V)
    base = ((4 * L.plane_stride + vol_pos(L, b, X, Y, Z)) * 8).reshape(-1)
    stale = torch.randint(-32768, 32768, (base.numel(), 8), generator=g, dtype=torch.int32).to(torch.int16)
    for e in range(8):
        flat[(base + e).cuda()] = stale[:, e].cuda()
    before = flat.cpu()
    grid = occ.cuda().contiguous()
    _lib.occ_expand_zwin(grid, buf, lay, 32)
    torch.cuda.synchronize()
    assert not bool(grid.any()), "occ_expand_zwin: the grid was not left all-zero"
    want = before.clone()
    one = storage_bits(torch.ones(1), f16)[0]
    for e in range(8):
        zz = Z + e - 3
        inside = (zz >= 0) & (zz < V)
        v = occ[b, X, Y, zz.clamp(0, V - 1)]
        want[base + e] = torch.where(inside & (v != 0), one, torch.zeros((), dtype=torch.int16)).reshape(-1)
    got = flat.cpu()
    bad = got != want
    assert not bool(bad.any()), f"occ_expand_zwin V{V} B{B}: {int(bad.sum())} elements differ, first {bad.nonzero()[:6, 0].tolist()}"


# ==== with_intersection product =========================================================================================
def _feature_bits(n, f16, g):
    """Random finite storage values with planted +-0, subnormals, the largest finite value, +-inf and NaN."""
    v = torch.randn(n, generator=g) * 4
    bits = storage_bits(v, f16)
    specials = ([0x0000, 0x8000, 0x0001, 0x8003, 0x03FF, 0x7BFF, 0xFBFF, 0x7C00, 0xFC00, 0x7E00] if f16 else
                [0x0000, 0x8000, 0x0001, 0x8003, 0x007F, 0x7F7F, 0xFF7F, 0x7F80, 0xFF80, 0x7FC0])
    sp = torch.tensor(specials, dtype=torch.int32).to(torch.int16)
    idx = torch.randint(0, n, (sp.numel() * 50,), generator=g)
    bits[idx] = sp.repeat(50)
    return bits


@pytest.mark.gpu
@pytest.mark.parametrize("S,B", [(16, 2), (24, 3), (64, 1)])
def test_intersect(S, B):
    """Planes 4-7 = storage rounding of fl32(x s) (bit for bit; NaN stays NaN; inf * 0 is NaN; the fp16 build
    saturates inf * 1 to 65504), planes 0-3 and the occupancy plane unchanged, every other cell and the spare frame
    keep their sentinel."""
    from sceneego_b200 import _lib
    f16 = _lib.act_dtype_name() == "f16"
    lay = _lib.vol_layout(S, 3, B + 1)
    L = model_layout("pad3", S, B + 1)
    buf = _lib.alloc_volume(lay, 72, "cuda")
    flat = buf.view(torch.int16).reshape(-1)
    flat.fill_(-1)
    g = torch.Generator().manual_seed(S + B)
    b, X, Y, Z = _grid(B, S)
    idx = {ch: elem_index(L, b, X, Y, Z, ch).reshape(-1) for ch in list(range(64)) + [64]}
    n = b.numel()
    feats = {ch: _feature_bits(n, f16, g) for ch in range(32)}
    occ = (torch.rand(n, generator=g) < 0.5).float()
    host = flat.cpu()
    for ch in range(32):
        host[idx[ch]] = feats[ch]
    host[idx[64]] = storage_bits(occ, f16)
    flat.copy_(host.cuda())
    _lib.intersect(buf, lay, B, 32)
    torch.cuda.synchronize()
    got = flat.cpu()
    want = host.clone()
    for ch in range(32):
        prod = decode_bits(feats[ch], f16) * occ
        want[idx[32 + ch]] = storage_bits(prod, f16)
    # bit for bit everywhere; only where the kernel stores a product may a NaN differ in its payload
    same = got == want
    written = torch.cat([idx[32 + ch] for ch in range(32)])
    nan_both = torch.isnan(decode_bits(want[written], f16)) & torch.isnan(decode_bits(got[written], f16))
    same[written] |= nan_both
    assert bool(same.all()), f"intersect S{S} B{B}: {int((~same).sum())} elements differ, first {(~same).nonzero()[:6, 0].tolist()}"


@pytest.mark.gpu
def test_intersection_input_matches_cat_of_live_planes():
    """The 65-channel V2V input as the network builds it for with_intersection=true from depth maps (unprojection
    into planes 0-3 with the planes behind cleared, voxelisation into channel 64, the product): planes 4-7 equal
    R16(vol * scene) and channel 64 the oracle's occupancy, element by element."""
    from oracle import sceneego_oracle as orc
    from sceneego_b200 import _lib
    from sceneego_b200.utils import synth
    V, B = 64, 2
    f16 = _lib.act_dtype_name() == "f16"
    tables = orc.StageTables(util.CALIB, V, 2.0)
    calib = _cam()
    lay = _lib.vol_layout(V, 3, B + 1)
    L = model_layout("pad3", V, B + 1)
    buf = _lib.alloc_volume(lay, 80, "cuda")
    buf.view(torch.int16).fill_(-1)
    feat = torch.randn(B, 64, 64, 32, generator=torch.Generator().manual_seed(2)).cuda()
    depth = synth.synthetic_depth_room(B, tables.ray, seed=5)
    _, grid = _lib.project_voxels(calib, V, 2.0, (IMG_H, IMG_W), "cuda")
    _lib.unproject(feat, grid, None, V, 2.0, IMG_H, IMG_W, None, buf, lay, extra_zero_planes=6)
    ray = _lib.ray_table(calib, "cuda")
    d = depth.reshape(B, depth.shape[-2], depth.shape[-1]).contiguous().float().cuda()
    _lib.voxelize_depth(d, ray, IMG_H, IMG_W, V, 2.0, None, buf, lay, channel=64)
    _lib.intersect(buf, lay, B, 32)
    torch.cuda.synchronize()
    flat = buf.view(torch.int16).reshape(-1).cpu()
    b, X, Y, Z = _grid(B, V)
    dh = depth.reshape(B, depth.shape[-2], depth.shape[-1]).numpy()
    scene = torch.from_numpy(np.stack([orc.voxelize_depth(dh[i], tables.ray, V, 2.0) for i in range(B)]))
    got_scene = decode_bits(flat[elem_index(L, b, X, Y, Z, 64)], f16)
    assert torch.equal(got_scene, scene), f"occupancy: {int((got_scene != scene).sum())} voxels differ from the oracle"
    for ch in range(32):
        vol = flat[elem_index(L, b, X, Y, Z, ch)]
        want = storage_bits(decode_bits(vol, f16) * scene, f16)
        got = flat[elem_index(L, b, X, Y, Z, 32 + ch)]
        assert torch.equal(got, want), f"channel {32 + ch}: {int((got != want).sum())} voxels differ"
    for ch in range(65, 80):
        assert not bool(flat[elem_index(L, b, X, Y, Z, ch)].any()), f"channel {ch} was not cleared"


# ==== CPU: the index model ===============================================================================================
@pytest.mark.parametrize("kind,S,B", [("plain", 16, 3), ("pad3", 64, 2), ("s2d", 64, 2), ("zwin", 48, 4), ("zwin", 8, 1)])
def test_index_model_matches_the_layout_maker(kind, S, B):
    """The model's pitches equal sceneego_vol_layout_make*; its element indices are distinct, inside the buffer and
    clear of every frame's guard and of the slack after the last frame."""
    from sceneego_b200 import _lib
    L = model_layout(kind, S, B)
    lay = (_lib.vol_layout_s2d(S, B) if kind == "s2d" else _lib.vol_layout_zwin(S, B) if kind == "zwin"
           else _lib.vol_layout(S, L.pad, B))
    for f in ("side", "pad", "pitch_y", "pitch_x", "guard", "frame_pitch", "plane_stride", "s2d", "zwin"):
        assert getattr(lay, f) == getattr(L, f), f
    b, X, Y, Z = _grid(B, S)
    nch = 33 if kind in ("s2d", "zwin") else 16
    idx = torch.cat([elem_index(L, b, X, Y, Z, ch).reshape(-1) for ch in range(nch)])
    assert idx.unique().numel() == idx.numel()
    pos = (idx // 8) % L.plane_stride
    assert bool((pos < B * L.frame_pitch).all()) and bool((pos % L.frame_pitch >= L.guard).all())


# ==== both storage builds ================================================================================================
@pytest.mark.gpu
@pytest.mark.skipif(F16_RUN, reason="already running on the fp16-storage build")
def test_exact_rest_with_fp16_storage_build():
    """The storage-dependent tests (layouts and the intersection) on libsceneego_b200_f16.so, in a subprocess."""
    env = dict(os.environ, SCENEEGO_ACT_DTYPE="f16", PYTHONPATH=util.ROOT)
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_exact_rest.py", "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider", "-k", "pack or unpack or occ_expand or intersect"],
                       cwd=util.ROOT, env=env, capture_output=True, text=True, timeout=1800)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert " passed" in tail.splitlines()[-1]

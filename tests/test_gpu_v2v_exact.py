"""Every V2V kernel element by element against a float64 reference of the same operation (tests/v2v_reference.py).

Two modes per case:
- "exact": integer data whose partial sums are all exact in fp32; the 16-bit output must equal R16(reference) bit for
  bit, for the tensor kernels and their CUDA-core checkers alike;
- "random": Gaussian data under a per-element bound (v2v_reference.assert_within).

Destinations are filled with 0xFFFF (NaN in bf16 and fp16) before the launch and the layouts hold one frame more than
the batch that runs: valid cells must hold the reference, pad and guard cells the sentinel or +0, the spare frame the
sentinel everywhere.  The CPU tests anchor the fold against the packer's blob and check the bound itself."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests import util
from tests import v2v_reference as vr

F64 = torch.float64
F16_RUN = os.environ.get("SCENEEGO_ACT_DTYPE", "bf16").lower() in ("f16", "fp16", "float16")
MODES = ["exact", "random"]


# ---- one-op programs over sentinel-filled destinations ------------------------------------------------------------
class Rig:
    """A throwaway single-op program.  Layouts are made for `frames` frames; destinations start as all-0xFFFF."""

    def __init__(self, frames, device="cuda"):
        from sceneego_b200.network.v2v import _Program
        pg = _Program.__new__(_Program)
        pg.side, pg.chunk, pg.device = 0, frames, torch.device(device)
        pg.ops, pg.buffers, pg.buf_level, pg.free, pg.blob_parts, pg.blob_bytes = [], [], [], {}, [], 0
        pg.flops, pg.meta = 0, []
        self.lays, self.sentinel = [], []
        pg.lay_of = lambda i: self.lays[i]
        self.pg, self.frames, self.device = pg, frames, torch.device(device)

    def volume(self, lay, channels, x=None, sentinel=False):
        from sceneego_b200 import _lib
        t = _lib.alloc_volume(lay, channels, self.device)
        if x is not None:
            _lib.pack_volume(x.to(self.device, torch.float32).contiguous(), t, lay)
        return self._add(t, lay, sentinel)

    def logits(self, channels, side):
        t = torch.empty(self.frames, channels, side, side, side, dtype=torch.float32, device=self.device)
        return self._add(t, None, True)

    def _add(self, t, lay, sentinel):
        self.pg.buffers.append(t)
        self.pg.buf_level.append(0)
        self.lays.append(lay)
        self.sentinel.append(sentinel)
        return len(self.pg.buffers) - 1

    def buf(self, i):
        return self.pg.buffers[i]

    def run(self, batch, impl=0):
        from sceneego_b200 import _lib
        pg = self.pg
        if not hasattr(pg, "op_array"):
            if not pg.blob_parts:                    # max-pool: no weights
                pg._append_blob(np.zeros(256, np.uint8))
            pg.finalize()
        for i, t in enumerate(pg.buffers):
            if self.sentinel[i]:
                if t.dtype == torch.float32:
                    t.fill_(float("nan"))
                else:
                    t.view(torch.int16).fill_(-1)
        pg.op_array[0].impl = impl
        lib = _lib.load_library()
        _lib._check(lib.sceneego_v2v_run(pg.op_array, 1, pg.buf_ptrs, C.c_void_p(pg.blob.data_ptr()), int(batch),
                                         _lib._stream()), "v2v_run")
        torch.cuda.synchronize()


def cell_positions(lay, B):
    S = lay.side
    i = torch.arange(S, dtype=torch.int64)
    pos = (torch.arange(B, dtype=torch.int64)[:, None, None, None] * lay.frame_pitch + lay.guard
           + i[None, :, None, None] * lay.pitch_x + i[None, None, :, None] * lay.pitch_y + i[None, None, None, :])
    return pos.reshape(-1)


def decode(buf, lay, B, channels):
    """Raw read of a planar volume: (B, channels, S, S, S) float64 of the stored 16-bit values."""
    S = lay.side
    flat = buf.permute(1, 0, 2).reshape(lay.plane_stride, -1)
    v = flat[cell_positions(lay, B).to(buf.device)][:, :channels]
    return v.reshape(B, S, S, S, channels).permute(0, 4, 1, 2, 3).to(F64)


def check_untouched(buf, lay, batch, where):
    """Outside the valid cells of the first `batch` frames: the sentinel or +0 (conv epilogues zero the pad rows they
    own); from frame `batch` on: the sentinel everywhere."""
    bits = buf.view(torch.int16).permute(1, 0, 2).reshape(lay.plane_stride, -1)
    valid = torch.zeros(lay.plane_stride, dtype=torch.bool, device=buf.device)
    valid[cell_positions(lay, batch).to(buf.device)] = True
    other = bits[~valid]
    ok = (other == -1) | (other == 0)
    if not bool(ok.all()):
        pos = (~valid).nonzero()[:, 0][(~ok).any(1)]
        raise AssertionError(f"{where}: {pos.numel()} pad / guard cells hold neither the sentinel nor +0, "
                             f"first positions {pos[:8].tolist()} (frame pitch {lay.frame_pitch}, guard {lay.guard})")
    spare = bits[batch * lay.frame_pitch:]
    if not bool((spare == -1).all()):
        pos = (spare != -1).any(1).nonzero()[:, 0] + batch * lay.frame_pitch
        raise AssertionError(f"{where}: {pos.numel()} cells of frames >= the batch were written, first {pos[:8].tolist()}")


def check_volume(rig, idx, batch, channels, ref, mode, where):
    lay = rig.lays[idx]
    got = decode(rig.buf(idx), lay, batch, channels)
    if mode == "exact":
        vr.assert_exact(got, ref, where, lay.pitch_y)
    else:
        vr.assert_within(got, ref, where, lay.pitch_y)
    check_untouched(rig.buf(idx), lay, batch, where)
    return got


def check_logits(rig, idx, batch, ref, mode, where):
    t = rig.buf(idx)
    got = t[:batch].to(F64)
    if mode == "exact":
        vr.assert_exact(got, ref, where)
    else:
        vr.assert_within(got, ref, where)
    assert bool(torch.isnan(t[batch:]).all()), f"{where}: logits of frames >= the batch were written"
    return got


# ---- operands ----------------------------------------------------------------------------------------------------
def _conv(mode, cin, cout, k, seed, transposed=False):
    return (vr.int_conv(cin, cout, k, seed, transposed) if mode == "exact"
            else vr.rand_conv(cin, cout, k, seed, transposed))


def _vol(mode, g, B, C_, S):
    return vr.int_volume(g, B, C_, S) if mode == "exact" else vr.rand_volume(g, B, C_, S)


def _res(mode, g, B, C_, S):
    return vr.int_residual(g, B, C_, S) if mode == "exact" else vr.rand_volume(g, B, C_, S)


def _exact(ref, mode):
    if mode == "exact":
        ref.grid = vr.INT_GRID
    return ref


# ---- conv_tc_kernel / conv_simt_kernel -------------------------------------------------------------------------
TC_CASES = [
    # cin, cout, k, S, B, pad_src, xs, pair, residual
    (32, 32, 3, 16, 2, 1, 1, 1, True),
    (32, 32, 3, 16, 3, 1, 2, 1, True),
    (32, 32, 3, 16, 3, 1, 2, 2, True),
    (32, 32, 3, 8, 3, 1, 4, 1, True),
    (32, 16, 3, 8, 2, 1, 4, 1, True),
    (16, 32, 3, 16, 2, 1, 1, 1, False),
    (64, 64, 3, 16, 5, 1, 1, 2, True),        # odd item count on CTA pairs: the last item is repeated
    (32, 64, 3, 8, 3, 1, 1, 2, False),
    (64, 128, 3, 8, 2, 1, 1, 1, True),
    (128, 128, 3, 2, 2, 1, 1, 1, True),
    (128, 128, 3, 3, 1, 1, 1, 1, True),
    (128, 128, 3, 4, 2, 1, 1, 1, False),
    (128, 128, 3, 6, 1, 1, 1, 1, True),
    (128, 128, 3, 8, 2, 1, 1, 1, True),
    (65, 16, 7, 32, 1, 3, 4, 1, False),       # with_intersection stem: cin padded to 80, five K steps
    (16, 32, 1, 16, 2, 1, 1, 1, False),
    (32, 32, 1, 16, 2, 1, 1, 1, True),
    (32, 15, 1, 16, 2, 1, 1, 1, False),
]


def _tc_id(c):
    return f"{c[0]}-{c[1]}-k{c[2]}-S{c[3]}-B{c[4]}-xs{c[6]}-pair{c[7]}" + ("-res" if c[8] else "")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", TC_CASES, ids=_tc_id)
def test_conv_tc(case, mode):
    cin, cout, k, S, B, pad_src, xs, pair, res = case
    from sceneego_b200 import _lib
    conv, bn = _conv(mode, cin, cout, k, seed=cin * 1000 + cout * 10 + k + S)
    g = torch.Generator().manual_seed(S * 31 + B)
    x = _vol(mode, g, B, cin, S)
    if cin == 65:                                    # features, features x occupancy, occupancy
        occ = (torch.rand(B, 1, S, S, S, generator=g) < 0.3).to(F64)
        x[:, 32:64] = x[:, :32] * occ
        x[:, 64:65] = occ
    r = _res(mode, g, B, cout, S) if res else None
    rig = Rig(B + 1)
    cp = vr._pad16(cout)
    s = rig.volume(_lib.vol_layout(S, pad_src, B + 1), vr._pad16(cin), x)
    d = rig.volume(_lib.vol_layout(S, 1, B + 1), cp, sentinel=True)
    ri = rig.volume(_lib.vol_layout(S, 1, B + 1), cp, r) if res else -1
    rig.pg.conv(conv, bn, s, d, relu=True, res=ri, xstack=xs, cta_pair=pair)
    ref = _exact(vr.conv_ref(x.cuda(), conv, bn, relu=True, res=r.cuda() if res else None, cout_pad=cp), mode)
    for impl, name in ((0, "conv_tc"), (1, "conv_simt")):
        rig.run(B, impl)
        check_volume(rig, d, B, cp, ref, mode, f"{name} {_tc_id(case)} {mode}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cout", [15, 16])
def test_conv_f32_output(cout, mode):
    """The unfused tail's last layer: a 1x1 conv writing f32 logits (B, cout_real, S, S, S), acc + b'."""
    from sceneego_b200 import _lib
    S, B = 16, 2
    conv, _ = _conv(mode, 32, cout, 1, seed=70 + cout)
    g = torch.Generator().manual_seed(cout)
    x = _vol(mode, g, B, 32, S)
    rig = Rig(B + 1)
    s = rig.volume(_lib.vol_layout(S, 1, B + 1), 32, x)
    d = rig.logits(cout, S)
    rig.pg.conv(conv, None, s, d, relu=False, out_f32=True)
    ref = _exact(vr.conv_ref(x.cuda(), conv, None, relu=False, out16=False), mode)
    for impl, name in ((0, "conv_tc"), (1, "conv_simt")):
        rig.run(B, impl)
        check_logits(rig, d, B, ref, mode, f"{name} f32-output 32->{cout} {mode}")


SHORTCUT_CASES = [(32, 16, 3, 2, 2), (64, 16, 2, 1, 2), (128, 8, 2, 1, 1), (32, 64, 1, 2, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("c,S,B,xs,pair", SHORTCUT_CASES)
def test_conv_tc_fused_shortcut(c, S, B, xs, pair, mode):
    """relu(bn(conv3(t)) + bn(conv1(x))) as one op on conv_tc_kernel; the bias is fl32(b_main + b_sc)."""
    from sceneego_b200 import _lib
    conv, bn = _conv(mode, c, c, 3, seed=3 * c + S)
    sc_conv, sc_bn = _conv(mode, c // 2, c, 1, seed=5 * c + S)
    g = torch.Generator().manual_seed(S + B + c)
    t_in, x_in = _vol(mode, g, B, c, S), _vol(mode, g, B, c // 2, S)
    rig = Rig(B + 1)
    lay = _lib.vol_layout(S, 1, B + 1)
    s = rig.volume(lay, c, t_in)
    d = rig.volume(lay, c, sentinel=True)
    s2 = rig.volume(lay, c // 2, x_in)
    rig.pg.conv(conv, bn, s, d, relu=True, xstack=xs, cta_pair=pair, shortcut=(sc_conv, sc_bn, s2))
    ref = _exact(vr.conv_ref(t_in.cuda(), conv, bn, relu=True, shortcut=(sc_conv, sc_bn, x_in.cuda())), mode)
    for impl, name in ((0, "conv_tc"), (1, "conv_simt")):
        rig.run(B, impl)
        check_volume(rig, d, B, c, ref, mode, f"{name} shortcut c{c} S{S} xs{xs} pair{pair} {mode}")


# ---- conv_march_kernel -----------------------------------------------------------------------------------------
MARCH_CASES = [
    # id, cin, cout, S, B, residual, shortcut, env
    ("32-S16", 32, 32, 16, 2, True, False, {}),
    ("16-S16", 16, 32, 16, 2, False, False, {}),
    ("32-S32", 32, 32, 32, 2, True, False, {}),
    ("32-S64", 32, 32, 64, 1, True, False, {}),
    ("32-S40-ring-wraps", 32, 32, 40, 2, True, False, {}),
    ("32-S32-B34-cut-ranges", 32, 32, 32, 34, True, False, {}),      # 306 items on 296 CTAs
    ("32-S16-B100-idle-ctas", 32, 32, 16, 100, True, False, {}),
    ("32-S16-B99-idle-ctas", 32, 32, 16, 99, False, False, {}),
    ("shortcut-S16", 32, 32, 16, 3, False, True, {}),
    ("shortcut-S32-B34", 32, 32, 32, 34, False, True, {}),
    ("32-S24-one-cta-per-sm", 32, 32, 24, 3, True, False, {"SCENEEGO_MARCH_CTAS": "1"}),
    ("32-S32-stages2", 32, 32, 32, 2, True, False, {"SCENEEGO_MARCH_STAGES": "2"}),
    ("shortcut-S16-stages2", 32, 32, 16, 3, False, True, {"SCENEEGO_MARCH_STAGES": "2"}),
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", MARCH_CASES, ids=[c[0] for c in MARCH_CASES])
def test_conv_march(case, mode, monkeypatch):
    name, cin, cout, S, B, res, sc, env = case
    from sceneego_b200 import _lib
    for k_, v_ in env.items():
        monkeypatch.setenv(k_, v_)
    conv, bn = _conv(mode, cin, cout, 3, seed=31 + cin + S + B)
    g = torch.Generator().manual_seed(S * 5 + B)
    x = _vol(mode, g, B, cin, S)
    rig = Rig(B + 1)
    lay = _lib.vol_layout(S, 1, B + 1)
    s = rig.volume(lay, cin, x)
    d = rig.volume(lay, cout, sentinel=True)
    r = x2 = None
    ri, shortcut = -1, None
    if res:
        r = _res(mode, g, B, cout, S)
        ri = rig.volume(lay, cout, r)
    if sc:
        sc_conv, sc_bn = _conv(mode, cin // 2, cout, 1, seed=78 + S)
        x2 = _vol(mode, g, B, cin // 2, S)
        shortcut = (sc_conv, sc_bn, rig.volume(lay, cin // 2, x2))
    rig.pg.conv(conv, bn, s, d, relu=True, res=ri, shortcut=shortcut, march=True)
    ref = _exact(vr.conv_ref(x.cuda(), conv, bn, relu=True, res=r.cuda() if res else None,
                             shortcut=(sc_conv, sc_bn, x2.cuda()) if sc else None), mode)
    for impl, kname in ((0, "conv_march"), (1, "conv_simt (marching blob)")):
        rig.run(B, impl)
        check_volume(rig, d, B, cout, ref, mode, f"{kname} {name} {mode}")


# ---- stems -------------------------------------------------------------------------------------------------------
def _stem_input(mode, g, B, V, density):
    x = _vol(mode, g, B, 33, V)
    x[:, 32] = (torch.rand(B, V, V, V, generator=g) < density).to(F64)       # occupancy is {0, 1}
    return x


def _stem_rig(kind, x, conv, bn, B, V, pair=1):
    from sceneego_b200 import _lib
    rig = Rig(B + 1)
    if kind == "march":
        s = rig.volume(_lib.vol_layout_zwin(V, B + 1), 40, x)
    else:
        s = rig.volume(_lib.vol_layout_s2d(V, B + 1), 33 * 8, x)
    d = rig.volume(_lib.vol_layout(V, 1, B + 1), 16, sentinel=True)
    if kind == "march":
        rig.pg.stem_march(conv, bn, s, d)
    else:
        rig.pg.stem_s2d(conv, bn, s, d, cta_pair=pair)
    return rig, d


STEM_CASES = [
    # V, B, occupancy density, SCENEEGO_STEM_SEGMENTS values (None: the launcher's choice)
    (16, 1, 0.1, (None, "32")),          # 32 segments at V = 16: the shortest segments the launcher allows
    (16, 3, 0.0, (None,)),
    (16, 5, 1.0, (None,)),
    (32, 1, 0.1, (None,)),
    (32, 3, 0.1, (None,)),
    (32, 5, 0.1, (None,)),
    (64, 1, 0.1, (None, "1", "7", "32")),  # 7: six segments of 10 planes and one of 4
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("V,B,density,segments", STEM_CASES)
def test_stem_march(V, B, density, segments, mode, monkeypatch):
    conv, bn = _conv(mode, 33, 16, 7, seed=5 + V)
    g = torch.Generator().manual_seed(V * 3 + B)
    x = _stem_input(mode, g, B, V, density)
    rig, d = _stem_rig("march", x, conv, bn, B, V)
    ref = _exact(vr.stem_ref(x.cuda(), conv, bn), mode)
    for seg in segments:
        if seg is None:
            monkeypatch.delenv("SCENEEGO_STEM_SEGMENTS", raising=False)
        else:
            monkeypatch.setenv("SCENEEGO_STEM_SEGMENTS", seg)
        rig.run(B, 0)
        check_volume(rig, d, B, 16, ref, mode, f"stem_march_tc V{V} B{B} occ{density} segments {seg} {mode}")
    monkeypatch.delenv("SCENEEGO_STEM_SEGMENTS", raising=False)
    rig.run(B, 1)
    check_volume(rig, d, B, 16, ref, mode, f"stem_march_simt V{V} B{B} {mode}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("pair", [1, 2])
@pytest.mark.parametrize("V,B", [(16, 2), (32, 1)])
def test_superseded_stem_s2d(V, B, pair, mode):
    """The space-to-depth stem (csrc/stem.cu), kept beside the marching stem."""
    conv, bn = _conv(mode, 33, 16, 7, seed=9 + V)
    g = torch.Generator().manual_seed(V + B + pair)
    x = _stem_input(mode, g, B, V, 0.2)
    rig, d = _stem_rig("s2d", x, conv, bn, B, V, pair)
    ref = _exact(vr.stem_ref(x.cuda(), conv, bn), mode)
    for impl, name in ((0, "stem_s2d_tc"), (1, "stem_s2d_simt")):
        rig.run(B, impl)
        check_volume(rig, d, B, 16, ref, mode, f"{name} V{V} B{B} pair{pair} {mode}")


# ---- transposed convs and max-pool -----------------------------------------------------------------------------
DECONV_CASES = [
    # cin, cout, S_in, B, skip
    (64, 32, 8, 2, True),          # npar 8
    (128, 64, 4, 2, True),         # npar 4
    (128, 128, 2, 2, True),        # npar 2
    (64, 32, 32, 1, True),         # 32^3 -> 64^3
    (128, 128, 3, 1, False),       # 3 -> 6
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cin,cout,S,B,skip", DECONV_CASES)
def test_deconv(cin, cout, S, B, skip, mode):
    """ConvTranspose3d(k2 s2) + BN: ReLU, then the skip."""
    from sceneego_b200 import _lib
    conv, bn = _conv(mode, cin, cout, 2, seed=11 + cin + cout + S, transposed=True)
    g = torch.Generator().manual_seed(4 + S + B)
    x = _vol(mode, g, B, cin, S)
    sk = _res(mode, g, B, cout, 2 * S) if skip else None
    rig = Rig(B + 1)
    s = rig.volume(_lib.vol_layout(S, 1, B + 1), cin, x)
    lay_d = _lib.vol_layout(2 * S, 1, B + 1)
    d = rig.volume(lay_d, cout, sentinel=True)
    ai = rig.volume(lay_d, cout, sk) if skip else -1
    rig.pg.deconv(conv, bn, s, d, add=ai)
    ref = _exact(vr.conv_ref(x.cuda(), conv, bn, relu=True, add_after=sk.cuda() if skip else None), mode)
    for impl, name in ((0, "deconv tensor path"), (1, "deconv2_kernel")):
        rig.run(B, impl)
        check_volume(rig, d, B, cout, ref, mode, f"{name} {cin}->{cout} S{S} {mode}")


@pytest.mark.gpu
@pytest.mark.parametrize("c,S,B", [(32, 64, 1), (64, 16, 2), (128, 6, 1), (128, 2, 2)])
def test_maxpool(c, S, B):
    from sceneego_b200 import _lib
    g = torch.Generator().manual_seed(c + S)
    x = vr.rand_volume(g, B, c, S)
    rig = Rig(B + 1)
    s = rig.volume(_lib.vol_layout(S, 1, B + 1), c, x)
    d = rig.volume(_lib.vol_layout(S // 2, 1, B + 1), c, sentinel=True)
    rig.pg.pool(s, d, c)
    rig.run(B)
    got = decode(rig.buf(d), rig.lays[d], B, c)
    assert torch.equal(got, F.max_pool3d(x.cuda(), 2, 2)), f"maxpool {c} {S}->{S // 2}"
    check_untouched(rig.buf(d), rig.lays[d], B, f"maxpool {c} {S}->{S // 2}")


# ---- fused tail ------------------------------------------------------------------------------------------------
def _tail_layers(mode, cout, seed):
    """Two Basic3DBlock(32, 32, 1) and Conv3d(32, cout, 1).  exact: weights k 2^-3 (|k| <= 3, then 1, 1), identity BN,
    biases exactly hi + lo with lo != 0 in both storage types (256 + 2^-3, 32 + 2^-6, 2 or 3 + 2^-10, random sign)."""
    from sceneego_b200.network.v2v import Basic3DBlock
    g = torch.Generator().manual_seed(seed)
    blocks = [Basic3DBlock(32, 32, 1).eval(), Basic3DBlock(32, 32, 1).eval()]
    out = nn.Conv3d(32, cout, 1).eval()
    convs = [blocks[0].block[0], blocks[1].block[0], out]
    bns = [blocks[0].block[1], blocks[1].block[1], None]
    if mode == "exact":
        for i, (cv, bn) in enumerate(zip(convs, bns)):
            n = cv.out_channels
            kmax = 3 if i == 0 else 1
            sign = torch.where(torch.rand(n, generator=g) < 0.75, 1.0, -1.0)
            base = [torch.full((n,), 256.0), torch.full((n,), 32.0),
                    torch.tensor([2.0, 3.0])[torch.randint(0, 2, (n,), generator=g)]][i]
            lo = [2.0 ** -3, 2.0 ** -6, 2.0 ** -10][i]
            with torch.no_grad():
                cv.weight.copy_(torch.randint(-kmax, kmax + 1, cv.weight.shape, generator=g).float() / 8)
                cv.bias.copy_(sign * (base + lo))
                if bn is not None:
                    bn.eps = 0.0
                    bn.weight.fill_(1.0)
                    bn.bias.zero_()
                    bn.running_mean.zero_()
                    bn.running_var.fill_(1.0)
    else:
        for i, (cv, bn) in enumerate(zip(convs, bns)):
            c2, b2 = vr.rand_conv(32, cv.out_channels, 1, seed + i)
            cv.load_state_dict(c2.state_dict())
            if bn is not None:
                bn.load_state_dict(b2.state_dict())
    return blocks, out, list(zip(convs, bns))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("cout", [1, 15, 16])
@pytest.mark.parametrize("impl", [0, 1, 2], ids=["tcgen05", "simt", "superseded-mma-sync"])
def test_tail(impl, cout, B, mode):
    """SCENEEGO_OP_TAIL_MLP: three chained 1x1 layers, hidden activations rounded after their ReLU."""
    from sceneego_b200 import _lib
    S = 16
    blocks, out, layers = _tail_layers(mode, cout, seed=cout * 10 + B)
    g = torch.Generator().manual_seed(B)
    x = _vol(mode, g, B, 32, S)
    rig = Rig(B + 1)
    s = rig.volume(_lib.vol_layout(S, 1, B + 1), 32, x)
    d = rig.logits(cout, S)
    rig.pg.tail_mlp(blocks, out, s, d)
    ref = vr.tail_ref(x.cuda(), layers, bias_hilo=impl == 0)
    if mode == "exact":
        ref.grid = 2.0 ** -10
    rig.run(B, impl)
    check_logits(rig, d, B, ref, mode, f"tail impl {impl} cout {cout} B{B} {mode}")


# ---- 16-bit range --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_outputs_beyond_the_storage_range():
    """Exact outputs far beyond 65504: the fp16 build stores exactly +-65504 (cvt.rn.satfinite), never inf; the bf16
    build stores R16 of the exact value."""
    from sceneego_b200 import _lib
    S, B = 8, 2
    conv, bn = vr.int_conv(128, 128, 3, seed=12)
    g = torch.Generator().manual_seed(12)
    x = vr.int_volume(g, B, 128, S, scale=4096.0)
    rig = Rig(B + 1)
    lay = _lib.vol_layout(S, 1, B + 1)
    s = rig.volume(lay, 128, x)
    d = rig.volume(lay, 128, sentinel=True)
    rig.pg.conv(conv, bn, s, d, relu=False)
    ref = vr.conv_ref(x.cuda(), conv, bn, relu=False)
    ref.grid = vr.INT_GRID * 4096
    assert float(ref.value.abs().max()) > 65504 * 4
    for impl in (0, 1):
        rig.run(B, impl)
        got = check_volume(rig, d, B, 128, ref, "exact", f"large outputs impl {impl}")
        if F16_RUN:
            assert float(got.abs().max()) == 65504.0 and bool(torch.isfinite(got).all())


@pytest.mark.gpu
def test_gpu_reference_matches_cpu_reference():
    """The float64 reference on the GPU equals the same computation on the CPU (integer data: bit for bit)."""
    S, B = 8, 2
    g = torch.Generator().manual_seed(8)
    conv, bn = vr.int_conv(32, 32, 3, seed=8)
    x, r = vr.int_volume(g, B, 32, S), vr.int_residual(g, B, 32, S)
    a = vr.conv_ref(x.cuda(), conv, bn, relu=True, res=r.cuda())
    b = vr.conv_ref(x, conv, bn, relu=True, res=r)
    assert torch.equal(a.value.cpu(), b.value)
    dc, dbn = vr.int_conv(64, 32, 2, seed=9, transposed=True)
    xd = vr.int_volume(g, B, 64, S // 2)
    assert torch.equal(vr.conv_ref(xd.cuda(), dc, dbn, relu=True).value.cpu(), vr.conv_ref(xd, dc, dbn, relu=True).value)
    sc, sbn = vr.int_conv(33, 16, 7, seed=10)
    xs = vr.int_volume(g, 1, 33, S)
    assert torch.equal(vr.stem_ref(xs.cuda(), sc, sbn).value.cpu(), vr.stem_ref(xs, sc, sbn).value)


# ---- every op of real programs, one at a time ------------------------------------------------------------------
def _recording(monkeypatch):
    """Wrap the _Program op builders so that each op remembers the modules it came from."""
    from sceneego_b200.network.v2v import _Program
    for name in ("conv", "deconv", "pool", "stem_march", "stem_s2d", "tail_mlp"):
        orig = getattr(_Program, name)

        def wrapped(self, *a, _orig=orig, _name=name, **kw):
            n = len(self.ops)
            _orig(self, *a, **kw)
            assert len(self.ops) == n + 1
            self.__dict__.setdefault("op_sources", []).append((_name, a, kw))
        monkeypatch.setattr(_Program, name, wrapped)


def _read_input(pg, idx, B, channels):
    from sceneego_b200 import _lib
    lay = pg.lay_of(idx)
    if lay.zwin or lay.s2d:
        return _lib.unpack_volume(pg.buffers[idx], lay, B, channels).to(F64)
    return decode(pg.buffers[idx], lay, B, channels)


def _op_ref(pg, op, src, B):
    """Reference of one program op from the live buffers it reads."""
    from sceneego_b200 import _lib
    kind, a, kw = src
    if kind == "pool":
        return "pool", F.max_pool3d(_read_input(pg, op.src, B, op.cin), 2, 2)
    if kind in ("stem_march", "stem_s2d"):
        return "conv", vr.stem_ref(_read_input(pg, op.src, B, 33), a[0], a[1])
    if kind == "tail_mlp":
        blocks, out = a[0], a[1]
        layers = [(b.block[0], b.block[1]) for b in blocks] + [(out, None)]
        return "tail", vr.tail_ref(_read_input(pg, op.src, B, 32), layers, bias_hilo=True)
    conv, bn = a[0], a[1]
    x = _read_input(pg, op.src, B, conv.in_channels)
    if kind == "deconv":
        skip = _read_input(pg, op.res, B, conv.out_channels) if op.flags & _lib.F_ADD_AFTER else None
        return "conv", vr.conv_ref(x, conv, bn, relu=True, add_after=skip)
    res = _read_input(pg, op.res, B, conv.out_channels) if op.flags & _lib.F_RESIDUAL else None
    shortcut = kw.get("shortcut")
    if shortcut is not None:
        shortcut = (shortcut[0], shortcut[1], _read_input(pg, shortcut[2], B, shortcut[0].in_channels))
    out_f32 = bool(op.flags & _lib.F_OUT_F32)
    return "conv", vr.conv_ref(x, conv, bn, relu=bool(op.flags & _lib.F_RELU), res=res, shortcut=shortcut,
                               out16=not out_f32, cout_pad=None if out_f32 else op.cout)


def _run_program_op_by_op(m, V, chunk, B, monkeypatch, seed=1):
    from sceneego_b200 import _lib
    from sceneego_b200.utils import synth
    sd = synth.synthetic_state_dict([(k, tuple(v.shape)) for k, v in m.state_dict().items()], seed=seed, mode="random_bn")
    m.load_state_dict(sd, strict=True)
    m.eval()
    _recording(monkeypatch)
    pg = m.program(V, chunk, "cuda")
    assert len(pg.op_sources) == len(pg.ops)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, m.input_channels, V, V, V, generator=g).abs()
    if m.input_channels == 33:
        x[:, 32] = (x[:, 32] > 1.0).float()
    _lib.pack_volume(x.cuda(), pg.buffers[pg.in_buf], pg.lay_in)
    logits = torch.full((chunk, m.output_channels, V, V, V), float("nan"), device="cuda")
    pg.buf_ptrs[pg.logits_buf] = C.c_void_p(logits.data_ptr())
    lib = _lib.load_library()
    checked = 0
    for i, (op, src) in enumerate(zip(pg.op_array, pg.op_sources)):
        kind, ref = _op_ref(pg, op, src, B)
        _lib._check(lib.sceneego_v2v_run(C.byref(op), 1, pg.buf_ptrs, C.c_void_p(pg.blob.data_ptr()), B,
                                         _lib._stream()), f"op {i}")
        torch.cuda.synchronize()
        where = f"op {i} ({src[0]}, type {op.type}, side {op.lay_src.side}, {op.cin}->{op.cout})"
        if kind == "pool":
            got = decode(pg.buffers[op.dst], pg.lay_of(op.dst), B, op.cout)
            assert torch.equal(got, ref), where
        elif kind == "tail" or op.flags & _lib.F_OUT_F32:
            got = logits[:B].to(F64)
            vr.assert_within(got, ref, where)
            assert bool(torch.isnan(logits[B:]).all()), f"{where}: logits of frames >= the batch were written"
        else:
            lay = pg.lay_of(op.dst)
            got = decode(pg.buffers[op.dst], lay, B, ref.value.shape[1])
            vr.assert_within(got, ref, where, lay.pitch_y)
        checked += 1
    assert checked == len(pg.ops)


def _variant(**kw):
    from sceneego_b200.network.v2v import V2VModel
    m = V2VModel(33, 15)
    for k_, v_ in kw.items():
        setattr(m, k_, v_)
    return m


PROGRAM_VARIANTS = {
    "default": {},
    "stem-s2d": {"stem": "s2d"},
    "no-march": {"march": False},
    "no-cta-pair": {"cta_pair": 1},
    "unfused-tail": {"fuse_tail": False},
    "unfused-shortcut": {"fuse_shortcut": False},
}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(PROGRAM_VARIANTS))
def test_program_ops_v32(variant, monkeypatch):
    _run_program_op_by_op(_variant(**PROGRAM_VARIANTS[variant]), 32, 2, 2, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("V", [64, 96])
def test_program_ops_large(V, monkeypatch):
    """V = 64, and V = 96 whose deepest levels are S = 6 and 3."""
    _run_program_op_by_op(_variant(), V, 1, 1, monkeypatch, seed=V)


@pytest.mark.gpu
def test_program_ops_intersection_input(monkeypatch):
    from sceneego_b200.network.v2v import V2VModel
    _run_program_op_by_op(V2VModel(65, 15), 32, 1, 1, monkeypatch, seed=3)


@pytest.mark.gpu
def test_program_ops_simple_model(monkeypatch):
    from sceneego_b200.network.v2v import V2VModelSimple
    _run_program_op_by_op(V2VModelSimple(33, 15), 32, 2, 2, monkeypatch, seed=4)


@pytest.mark.gpu
def test_program_ops_batch_below_chunk(monkeypatch):
    """A program built for 4 frames run with 3, as V2VModel.program does when it reuses a larger pool."""
    _run_program_op_by_op(_variant(), 32, 4, 3, monkeypatch, seed=5)


# ---- both storage builds -----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.skipif(F16_RUN, reason="already running on the fp16-storage build")
def test_v2v_exact_with_fp16_storage_build():
    """This file's GPU tests on libsceneego_b200_f16.so (one activation dtype per process: a subprocess)."""
    env = dict(os.environ, SCENEEGO_ACT_DTYPE="f16", PYTHONPATH=util.ROOT)
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_v2v_exact.py", "-m", "gpu", "-x", "-q",
                        "-p", "no:cacheprovider"], cwd=util.ROOT, env=env, capture_output=True, text=True, timeout=1800)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert " passed" in tail.splitlines()[-1]


# ---- CPU: the fold equals the packer, and the bound is neither vacuous nor flaky ---------------------------------
def _decode_blob(w_out):
    return torch.from_numpy(np.ascontiguousarray(w_out).view(np.int16)).view(vr.storage_dtype())


@pytest.mark.parametrize("k,transposed,cin,cout", [(3, False, 32, 32), (1, False, 32, 15), (7, False, 33, 16),
                                                    (3, False, 16, 64), (2, True, 64, 32), (2, True, 128, 128)])
def test_fold_equals_packer(k, transposed, cin, cout):
    """sceneego_v2v_pack_conv (xs = 1, n_split = 1) decoded: weights and biases equal this file's fold bit for bit,
    including a weight beyond the fp16 range (saturates to 65504 on the fp16 build)."""
    from sceneego_b200.network.v2v import _Program
    conv, bn = vr.rand_conv(cin, cout, k, seed=cin + cout + k, transposed=transposed)
    with torch.no_grad():
        conv.weight.view(-1)[5] = 1.0e6
        conv.weight.view(-1)[6] = -3.0e5
    cin_p, cout_p = vr._pad16(cin), vr._pad16(cout)
    pg = _Program.__new__(_Program)
    w_out, b_out = pg.pack_arrays(conv, bn, cin_p, cout_p)
    wf, bf = vr.fold(conv, bn)
    taps = k ** 3
    blob = _decode_blob(w_out)
    if transposed:
        npar = min(8, 256 // cout_p)
        got = blob.view(8 // npar, cin_p // 8, npar, cout_p, 8).permute(1, 4, 3, 0, 2).reshape(cin_p, cout_p, taps)
        got = got[:cin, :cout].reshape(wf.shape)
    else:
        got = blob.view(taps, cin_p // 8, cout_p, 8).permute(2, 1, 3, 0).reshape(cout_p, cin_p, taps)
        assert not bool(got[cout:].to(F64).any()) and not bool(got[:, cin:].to(F64).any())
        got = got[:cout, :cin].reshape(wf.shape)
    want = wf.to(vr.storage_dtype())
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))
    assert torch.equal(torch.from_numpy(b_out[:cout]).to(F64), bf)
    assert not b_out[cout:].any()


def test_fused_shortcut_bias_equals_program():
    """_Program.conv's fused-shortcut bias is fl32(fl64(b_main) + fl64(b_sc))."""
    from sceneego_b200.network.v2v import _Program
    conv, bn = vr.rand_conv(32, 32, 3, seed=1)
    sc, sbn = vr.rand_conv(16, 32, 1, seed=2)
    pg = _Program.__new__(_Program)
    _, b1 = pg.pack_arrays(conv, bn, 32, 32)
    _, b2 = pg.pack_arrays(sc, sbn, 16, 32)
    want = (b1.astype(np.float64) + b2.astype(np.float64)).astype(np.float32)
    got = vr.fold_bias_sum(vr.fold(conv, bn)[1], vr.fold(sc, sbn)[1])
    assert torch.equal(got, torch.from_numpy(want).to(F64))


@pytest.mark.skipif(F16_RUN, reason="already running on the fp16-storage build")
def test_fold_equals_packer_on_fp16_build():
    env = dict(os.environ, SCENEEGO_ACT_DTYPE="f16", PYTHONPATH=util.ROOT)
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_v2v_exact.py", "-q", "-x", "-p", "no:cacheprovider",
                        "-k", "fold or bound or hilo"], cwd=util.ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-1500:]


def test_hilo_split_is_exact_for_the_exact_mode_biases():
    for b in (256.125, 32 + 2.0 ** -6, 2 + 2.0 ** -10, 3 + 2.0 ** -10):
        t = torch.tensor([b, -b], dtype=F64)
        assert torch.equal(vr.hilo(t), t)
        assert not torch.equal(vr.r16(t), t)         # lo != 0


def _bound_case():
    S, B = 16, 2
    conv, bn = vr.rand_conv(32, 32, 3, seed=21)
    g = torch.Generator().manual_seed(22)
    x, r = vr.rand_volume(g, B, 32, S), vr.rand_volume(g, B, 32, S)
    return conv, bn, x, r, vr.conv_ref(x, conv, bn, relu=True, res=r)


def test_bound_admits_an_fp32_conv_in_any_order():
    conv, bn, x, r, ref = _bound_case()
    for seed in range(3):
        got = vr.simulate_conv_f32(x, conv, bn, res=r, seed=seed)
        bad = ~vr.within_mask(got, ref)
        assert not bool(bad.any()), vr.localise(bad, f"fp32 conv, order {seed}", got, ref.value)


def test_bound_rejects_a_dropped_tap():
    conv, bn, x, r, ref = _bound_case()
    S = x.shape[-1]
    every = torch.ones(x.shape[0], S, S, S, dtype=torch.bool)
    got = vr.simulate_conv_f32(x, conv, bn, res=r, drop=(5, 13, every))
    frac = float((~vr.within_mask(got, ref)).to(F64).mean())
    assert frac >= 0.10, f"dropping one tap of one channel fails only {frac:.3f} of the elements"
    plane = torch.zeros_like(every)
    plane[:, ::8] = True
    got = vr.simulate_conv_f32(x, conv, bn, res=r, drop=(5, 13, plane))
    assert int((~vr.within_mask(got, ref)).sum()) > 0

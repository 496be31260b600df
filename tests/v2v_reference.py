"""Float64 references of the V2V ops, computed from exactly the operands the kernels see.

The fold is the host packers' (`sceneego_v2v_pack_conv`): scale = gamma / sqrt(var + eps) and shift = beta - mean * scale
in fp64 from the fp32 parameters, w' = R16(fl32(w * scale)), b' = fl32(bias * scale + shift).  R16 is round-to-nearest-
even to the 16-bit storage type (saturating at +-65504 on the fp16 build).  Each op is then evaluated in float64 with
the kernels' epilogue order.

Two ways to compare a kernel's output with a reference:
- integer data (`int_conv`, `int_volume`): every partial sum is exact in fp32, so the kernel's result does not depend on
  the order of summation and must equal R16(reference) bit for bit (`assert_exact`);
- random data: a per-element bound (`assert_within`),
  |got - ref| <= u16 (|ref| + E) + E + tau,  E = K 2^-23 A + 2^-23 (|acc| + |b'| + |r|),
  with A = sum |w'| |x| (one more conv of absolute values), K the padded reduction length, u16 the storage type's unit
  roundoff and tau its smallest subnormal.
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

F64 = torch.float64
EPS32 = 2.0 ** -23


def _pad16(c):
    return (c + 15) // 16 * 16


def storage_dtype():
    from sceneego_b200 import _lib
    return _lib.act_torch_dtype()


def u16():
    """Unit roundoff of the storage type: 2^-8 for bf16, 2^-11 for fp16."""
    return 2.0 ** -11 if storage_dtype() == torch.float16 else 2.0 ** -8


def tau():
    """Smallest positive subnormal of the storage type."""
    return 2.0 ** -24 if storage_dtype() == torch.float16 else 2.0 ** -133


def r16(t):
    """Round to fp32, then to the storage type (RNE; fp16 saturates like cvt.rn.satfinite); returned as float64."""
    t = t.to(torch.float32)
    if storage_dtype() == torch.float16:
        t = t.clamp(-65504.0, 65504.0)
    return t.to(storage_dtype()).to(F64)


# ---- the fold ----------------------------------------------------------------------------------------------------
def fold(conv, bn):
    """(w', b') of Conv3d / ConvTranspose3d + optional eval BatchNorm3d, as float64 CPU tensors (w' in the module's
    weight shape, b' of length out_channels)."""
    transposed = isinstance(conv, nn.ConvTranspose3d)
    w = conv.weight.detach().to("cpu", torch.float32).to(F64)
    cout = conv.out_channels
    b = conv.bias.detach().to("cpu", torch.float32).to(F64) if conv.bias is not None else torch.zeros(cout, dtype=F64)
    if bn is None:
        scale, shift = torch.ones(cout, dtype=F64), torch.zeros(cout, dtype=F64)
    else:
        g, bt, mu, var = (t.detach().to("cpu", torch.float32).to(F64)
                          for t in (bn.weight, bn.bias, bn.running_mean, bn.running_var))
        scale = g / torch.sqrt(var + float(bn.eps))
        shift = bt - mu * scale
    sc = scale.view(1, -1, 1, 1, 1) if transposed else scale.view(-1, 1, 1, 1, 1)
    return r16(w * sc), (b * scale + shift).to(torch.float32).to(F64)


def fold_bias_sum(b_main, b_sc):
    """Bias of a fused 1x1 projection shortcut: fl32(fl64(b_main) + fl64(b_sc))."""
    return (b_main + b_sc).to(torch.float32).to(F64)


def hilo(b):
    """The tcgen05 tail's bias as two 16-bit parts: hi = R16(b), lo = R16(fl32(b - hi)); returns hi + lo."""
    hi = r16(b)
    return hi + r16((b.to(torch.float32) - hi.to(torch.float32)).to(F64))


# ---- float64 evaluation ------------------------------------------------------------------------------------------
def _direct():
    # cuDNN may pick FFT or Winograd algorithms for float64, whose results are not exact sums: the reference uses
    # torch's own im2col + GEMM path
    return torch.backends.cudnn.flags(enabled=False)


def conv3d(x, w):
    """'Same' 3D convolution in float64 (odd k), in x-slabs so that the unfolded columns stay small."""
    k = w.shape[-1]
    r = k // 2
    S = x.shape[2]
    w = w.to(x.device)
    if k == 1:
        return torch.einsum("bcxyz,oc->boxyz", x, w.reshape(w.shape[0], w.shape[1]))
    xp = F.pad(x, (r, r, r, r, r, r))
    per_plane = x.shape[0] * x.shape[1] * k ** 3 * (S + 2 * r) ** 2 * 8
    step = max(1, min(S, (1 << 30) // max(per_plane, 1)))
    with _direct():
        return torch.cat([F.conv3d(xp[:, :, x0:min(S, x0 + step) + 2 * r], w) for x0 in range(0, S, step)], dim=2)


def conv_transpose3d(x, w):
    with _direct():
        return F.conv_transpose3d(x, w.to(x.device), stride=2)


class Ref:
    """Exact value of an op's output (float64, before the output rounding) and the radius E of the bound."""

    def __init__(self, value, radius, out16=True, grid=None, absum=None):
        self.value, self.radius, self.out16 = value, radius, out16
        self.grid, self.absum = grid, absum      # integer mode: every partial sum is a multiple of `grid`, below absum


def conv_ref(x, conv, bn, relu, res=None, add_after=None, shortcut=None, out16=True, cout_pad=None):
    """Conv3d / ConvTranspose3d (k2 s2) + BN with the kernels' epilogue: t = acc + b'; + r if residual; ReLU;
    + r if added after.  shortcut = (conv1x1, bn, x2) accumulates into the same sum.  Channels up to cout_pad (zero
    weights and bias) are included, as the kernels write them."""
    transposed = isinstance(conv, nn.ConvTranspose3d)
    wf, bf = fold(conv, bn)
    op = conv_transpose3d if transposed else conv3d
    k = conv.kernel_size[0]
    acc, A = op(x, wf), op(x.abs(), wf.abs())
    K = _pad16(conv.in_channels) * (1 if transposed else k ** 3)
    if shortcut is not None:
        sc_conv, sc_bn, x2 = shortcut
        w2, b2 = fold(sc_conv, sc_bn)
        acc, A = acc + conv3d(x2, w2), A + conv3d(x2.abs(), w2.abs())
        K += _pad16(sc_conv.in_channels)
        bf = fold_bias_sum(bf, b2)
    b = bf.to(x.device).view(1, -1, 1, 1, 1)
    t = acc + b
    r = res if res is not None else add_after
    if res is not None:
        t = t + res
    if relu:
        t = t.clamp_min(0)
    if add_after is not None:
        t = t + add_after
    E = K * EPS32 * A + EPS32 * (acc.abs() + b.abs() + (r.abs() if r is not None else 0))
    absum = A + b.abs() + (r.abs() if r is not None else 0)
    if cout_pad is not None and cout_pad > t.shape[1]:
        padc = (0, 0, 0, 0, 0, 0, 0, cout_pad - t.shape[1])
        t, E, absum = F.pad(t, padc), F.pad(E, padc), F.pad(absum, padc)
    return Ref(t, E, out16, absum=absum)


def stem_ref(x, conv, bn):
    """7^3 33 -> 16 stem + BN + ReLU (any of its kernels); K = 48 * 343 also covers the z-window occupancy plane's
    8 entries per tap."""
    return conv_ref(x, conv, bn, relu=True)


def tail_ref(x, layers, bias_hilo=False):
    """Two 1x1 conv + BN + ReLU layers and the 1x1 output conv, f32 logits.  Each hidden activation is rounded with R16
    after its ReLU; the radius of the hidden layers propagates (the next layer's E gains |W| e_prev).  bias_hilo: the
    bias enters as hi + lo (tail_tc_kernel), exact to u16^2 |b|."""
    h, e = x, None
    absum = None
    for i, (conv, bn) in enumerate(layers):
        wf, bf = fold(conv, bn)
        b = bf.to(x.device).view(1, -1, 1, 1, 1)
        acc, A = conv3d(h, wf), conv3d(h.abs(), wf.abs())
        t = acc + b
        E = 32 * EPS32 * A + EPS32 * (acc.abs() + b.abs())
        if bias_hilo:
            E = E + u16() ** 2 * b.abs()
        if e is not None:
            E = E + conv3d(e, wf.abs())
        absum = A + b.abs()
        if i < len(layers) - 1:
            t = t.clamp_min(0)
            e = E + u16() * (2 * t.abs() + E) + 2 * tau()
            h = r16(t)
    return Ref(t, E, out16=False, absum=absum)


# ---- comparisons -------------------------------------------------------------------------------------------------
def localise(bad, where, got=None, want=None, pitch_y=None, limit=8):
    """Summary of wrong elements of a (B, C, S, S, S) mask: count, first coordinates, histograms by x-plane, by
    128-cell tile of the (y, z) plane, by frame and by 8-channel group."""
    idx = bad.nonzero()
    n = idx.shape[0]
    lines = [f"{where}: {n} of {bad.numel()} elements wrong"]
    for row in idx[:limit].tolist():
        s = f"  (b, c, x, y, z) = {tuple(row)}"
        if got is not None:
            s += f": got {got[tuple(row)].item()!r}, want {want[tuple(row)].item()!r}"
        lines.append(s)
    S = bad.shape[-1]
    py = pitch_y or S
    tiles = (idx[:, 3] * py + idx[:, 4]) // 128

    def hist(col, name):
        v, c = torch.unique(col, return_counts=True)
        lines.append(f"  by {name}: " + ", ".join(f"{a}:{b}" for a, b in zip(v.tolist()[:40], c.tolist()[:40])))
    hist(idx[:, 2], "x-plane")
    hist(tiles, "(y,z) tile of 128 cells")
    hist(idx[:, 0], "frame")
    hist(idx[:, 1] // 8, "8-channel group")
    return "\n".join(lines)


def assert_exact(got, ref, where, pitch_y=None):
    """Integer data: the output equals R16(reference) (f32 outputs: the reference itself), value for value."""
    if ref.absum is not None and ref.grid is not None:
        # the premise of bit-exactness: every partial sum is a multiple of `grid` below 2^24 grid
        assert float(ref.absum.max()) < 2.0 ** 24 * ref.grid, f"{where}: operands too large for exact fp32 sums"
    want = r16(ref.value) if ref.out16 else ref.value
    got = got.to(F64)
    bad = ~(got == want)
    if bool(bad.any()):
        raise AssertionError(localise(bad, where, got, want, pitch_y))


def within_mask(got, ref):
    got = got.to(F64)
    E = ref.radius
    lim = (u16() * (ref.value.abs() + E) + E + tau()) if ref.out16 else E + 2.0 ** -149
    return torch.isfinite(got) & ((got - ref.value).abs() <= lim)


def assert_within(got, ref, where, pitch_y=None):
    bad = ~within_mask(got, ref)
    if bool(bad.any()):
        raise AssertionError(localise(bad, where, got.to(F64), ref.value, pitch_y))


# ---- operands ----------------------------------------------------------------------------------------------------
def int_volume(g, B, C, S, lo=-2, hi=2, scale=1.0):
    return torch.randint(lo, hi + 1, (B, C, S, S, S), generator=g).to(F64) * scale


def int_residual(g, B, C, S):
    """Multiples of 2^-3 in [-4, 4]."""
    return torch.randint(-32, 33, (B, C, S, S, S), generator=g).to(F64) / 8


def _set_int_bn(bn, g):
    c = bn.num_features
    bn.eps = 0.0
    with torch.no_grad():
        bn.running_var.copy_(torch.tensor([1.0, 4.0])[torch.randint(0, 2, (c,), generator=g)])
        bn.weight.copy_(torch.tensor([0.5, 1.0, 2.0])[torch.randint(0, 3, (c,), generator=g)])
        bn.bias.copy_(torch.randint(-32, 33, (c,), generator=g).float() / 32)
        bn.running_mean.copy_(torch.randint(-32, 33, (c,), generator=g).float() / 32)


def int_conv(cin, cout, k, seed, transposed=False, kmax=7, with_bn=True):
    """Conv (+ BN) whose fold is exact: weights k 2^-5 (|k| <= kmax), biases, beta and mean multiples of 2^-5, eps = 0,
    var in {1, 4} and gamma in {0.5, 1, 2} (the scale is a power of two).  Folded weights and biases are multiples of
    2^-7, so with integer inputs every partial sum is a multiple of 2^-7."""
    g = torch.Generator().manual_seed(seed)
    conv = (nn.ConvTranspose3d(cin, cout, 2, stride=2) if transposed else nn.Conv3d(cin, cout, k, padding=(k - 1) // 2))
    with torch.no_grad():
        conv.weight.copy_(torch.randint(-kmax, kmax + 1, conv.weight.shape, generator=g).float() / 32)
        conv.bias.copy_(torch.randint(-32, 33, (cout,), generator=g).float() / 32)
    bn = None
    if with_bn:
        bn = nn.BatchNorm3d(cout)
        _set_int_bn(bn, g)
        bn.eval()
    return conv.eval(), bn


INT_GRID = 2.0 ** -7


def rand_conv(cin, cout, k, seed, transposed=False):
    """Gaussian conv + BN drawn like tests/test_gpu_v2v._mk_conv (CPU modules)."""
    g = torch.Generator().manual_seed(seed)
    conv = (nn.ConvTranspose3d(cin, cout, 2, stride=2) if transposed else nn.Conv3d(cin, cout, k, padding=(k - 1) // 2))
    bn = nn.BatchNorm3d(cout)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) * (2.0 / (cin * k ** 3)) ** 0.5)
        conv.bias.copy_(torch.randn(cout, generator=g) * 0.1)
        bn.weight.copy_(torch.rand(cout, generator=g) + 0.5)
        bn.bias.copy_(torch.randn(cout, generator=g) * 0.1)
        bn.running_mean.copy_(torch.randn(cout, generator=g) * 0.1)
        bn.running_var.copy_(torch.rand(cout, generator=g) * 1.5 + 0.5)
    return conv.eval(), bn.eval()


def rand_volume(g, B, C, S):
    """Gaussian data rounded to the storage type."""
    return r16(torch.randn(B, C, S, S, S, generator=g).to(F64))


def simulate_conv_f32(x, conv, bn, res=None, relu=True, drop=None, seed=0):
    """CPU model of a kernel: the folded operands summed in fp32 in a shuffled channel order, the fp32 epilogue, the
    output rounded to the storage type.  drop = (ci, tap, mask): zero tap `tap` of input channel ci where `mask`
    (B, S, S, S) is true (a kernel that skips it there)."""
    wf, bf = fold(conv, bn)
    perm = torch.randperm(x.shape[1], generator=torch.Generator().manual_seed(seed))
    w32 = wf[:, perm].to(torch.float32)
    acc = F.conv3d(x[:, perm].to(torch.float32), w32, padding=wf.shape[-1] // 2)
    if drop is not None:
        ci, tap, mask = drop
        k = wf.shape[-1]
        wt = torch.zeros_like(wf[:, :1]).to(torch.float32)
        wt.view(wt.shape[0], -1)[:, tap] = wf[:, ci].reshape(wf.shape[0], -1)[:, tap].to(torch.float32)
        part = F.conv3d(x[:, ci:ci + 1].to(torch.float32), wt, padding=k // 2)
        acc = acc - part * mask[:, None].to(torch.float32)
    t = acc + bf.to(torch.float32).view(1, -1, 1, 1, 1)
    if res is not None:
        t = t + res.to(torch.float32)
    if relu:
        t = t.clamp_min(0)
    return r16(t)

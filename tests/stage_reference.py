"""Float64 references of the stage's non-V2V kernels, computed from exactly the operands the kernels see.

Kernels covered: the backbone hand-off (csrc/handoff.cu), the 1x1 feature conv (csrc/feature_conv.cu and its CUDA-core
form in csrc/geometry.cu), the unprojection and the generic grid_sample (csrc/geometry.cu) and the soft-argmax
(csrc/softargmax.cu).  R16, u16, tau and the comparisons come from tests/v2v_reference.py.

Bounds (u = 2^-24, the fp32 unit roundoff; a tensor-core accumulation is charged 2u per addition):

- hand-off, GEMM 1 (deconv k4 s2 + BN, K1 = 4 taps x 256 channels):
    E1 = K1 2u A1 + 2u (|acc1| + |shift|),  A1 = sum |w'| |x|;
  the hidden activation is R16(ReLU(t1)), so its radius grows to e = E1 + u16 (2 |t1| + E1) + 2 tau;
  GEMM 2 (1x1, K2 = 256):  E2 = K2 2u A2 + 2u (|acc2| + |b2|) + sum |w2| e,  A2 = sum |w2| |h|  (as tail_ref).
- 1x1 feature conv on tensor cores: x = xh + xl + ex with xh = bf16(x), xl = bf16(x - xh), |ex| <= 2^-18 |x| (w alike);
  x w - (xh wh + xl wh + xh wl) = xl wl + ex w + (xh + xl) ew, at most 3.1 2^-18 |x| |w|; the three products are
  summed on the tensor core (768 additions) and the bias added in fp32:
    E = (3.1 2^-18 + 770 2u) A + u (|acc| + |b|),  A = sum |x| |w|;
  the CUDA-core kernel is a chain of 256 fmaf:  E = 256 u A + u (|acc| + |b|).
- bilinear sampling (unprojection, grid_sample): ix, iy are the kernel's fp32 values (emulated in NumPy float32), the
  exact weights are wx1 = ix - floor(ix), wx0 = 1 - wx1 (likewise y).  The kernel's wx0, wx1 are each within u of the
  exact ones, wx wy is rounded once (u), taps that share a source cell are merged (u each) and the at most four
  products are accumulated with fmaf or adds (4u of the running sum):
    E = sum_t |v_t| (8 u |w_t| + 3 u),  over the four taps t with their exact weights w_t and image values v_t.
- soft-argmax, softmax on: d_k = x_k mult - max(x mult).  The kernel evaluates exp2f((fl(x_k mult) - m) log2e): the
  product, the subtraction and the product with the fp32 log2e each round, so the exponent is off by at most
  u (|x_k mult| + 3 |d_k|) (natural units); exp2f adds 2 ulp (2^-22).  delta_k = 1.01 u (|x_k mult| + 3 |d_k|) + 2^-22
  bounds the relative error of one weight.  On its way into the sum s a weight passes through at most
  Ka = 4 iters + 5 + 8 + splits additions (u each: four per iteration of 4096 voxels in a thread, then the warp, block and
  split merges) and Km = iters + 5 + 8 + splits rescalings by exp2f((m_old - m_new) log2e), whose argument
  is at most D = max - min of x mult (5u + 3u D each: exp2f, the product, the argument rounding):
    path = Ka u + Km u (5 + 3 D),  rel_s = sum_k p_k delta_k + path;
    volume:   |o_k - p_k| <= 1.01 p_k (delta_k + rel_s + 2^-23) + 2^-147;
    keypoint: |kp - sum p c| <= 1.01 (sum_k p_k |c_k| (delta_k + path) + |kp| (rel_s + 2^-22)).
  softmax off: the volume is fl32(max(x mult, 0)) bit for bit; the keypoint is sum w c with
    E = (Ka + 1) u sum w |c|.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

from tests import v2v_reference as vr

F64 = torch.float64
U32 = 2.0 ** -24


# ---- backbone hand-off -------------------------------------------------------------------------------------------
def handoff_fold(deconv_w, gamma, beta, mean, var, eps):
    """(w1', shift) of ConvTranspose2d(256, 256, 4) + eval BatchNorm2d as the packer folds them: scale = gamma /
    sqrt(var + eps) in fp64, w1' = R16(fl32(w scale)) (cin, cout, 4, 4), shift = fl32(beta - mean scale)."""
    f = lambda t: t.detach().to("cpu", torch.float32).to(F64)
    scale = f(gamma) / torch.sqrt(f(var) + float(eps))
    w1 = vr.r16((f(deconv_w) * scale.view(1, -1, 1, 1)).to(torch.float32).to(F64))
    shift = (f(beta) - f(mean) * scale).to(torch.float32).to(F64)
    return w1, shift


def _deconv(x, w):
    with vr._direct():
        return F.conv_transpose2d(x, w.to(x.device), stride=2, padding=1)


def handoff_ref(x, w1, shift, w2, b2):
    """x (B, 256, h, w) float64 of R16 values, w1 (256, 256, 4, 4) folded, w2 (32, 256) R16, b2 (32,) ->
    Ref of (B, 2h, 2w, 32): ReLU(fl32(acc1 + shift)) -> R16 -> 1x1 -> acc2 + b2.  Ref.A holds both GEMMs'
    sum |w| |x| (for the integer-data precondition) as (A1, A2)."""
    dev = x.device
    sh = shift.to(dev).view(1, -1, 1, 1)
    acc1, A1 = _deconv(x, w1), _deconv(x.abs(), w1.abs())
    t1 = (acc1 + sh).clamp_min(0)
    E1 = 1024 * 2 * U32 * A1 + 2 * U32 * (acc1.abs() + sh.abs())
    e = E1 + vr.u16() * (2 * t1.abs() + E1) + 2 * vr.tau()
    h = vr.r16(t1)
    w2 = w2.to(dev)
    mm = lambda a, w: torch.einsum("bchw,oc->bhwo", a, w)
    acc2, A2 = mm(h, w2), mm(h.abs(), w2.abs())
    b = b2.to(dev).view(1, 1, 1, -1)
    E2 = 256 * 2 * U32 * A2 + 2 * U32 * (acc2.abs() + b.abs()) + mm(e, w2.abs())
    ref = vr.Ref(acc2 + b, E2, out16=False)
    ref.A = (A1, A2)
    return ref


def simulate_handoff(x, w1, shift, w2, b2, seed=0, drop=None):
    """CPU model of the kernel: both GEMMs in fp32 over a shuffled channel order, the hidden layer rounded with R16
    after the fp32 ReLU.  drop = (ci, ky, kx): that deconv tap of input channel ci is skipped."""
    g = torch.Generator().manual_seed(seed)
    p1 = torch.randperm(x.shape[1], generator=g)
    w1f = w1.clone()
    if drop is not None:
        ci, ky, kx = drop
        w1f[ci, :, ky, kx] = 0
    acc = F.conv_transpose2d(x[:, p1].float(), w1f[p1].float(), stride=2, padding=1)
    h = vr.r16((acc + shift.float().view(1, -1, 1, 1)).clamp_min(0))
    p2 = torch.randperm(h.shape[1], generator=g)
    out = torch.einsum("bchw,oc->bhwo", h[:, p2].float(), w2[:, p2].float()) + b2.float()
    return out.to(F64)


# ---- 1x1 feature conv --------------------------------------------------------------------------------------------
def bf16_split(t):
    """(hi, lo) of the kernel's split, as float64: hi = bf16(t), lo = bf16(fl32(t - hi))."""
    t = t.to(torch.float32)
    hi = t.to(torch.bfloat16).to(torch.float32)
    lo = (t - hi).to(torch.bfloat16).to(torch.float32)
    return hi.to(F64), lo.to(F64)


def feature_conv_ref(x, w, b, tensor_core=True):
    """x (B, 256, h, w), w (32, 256), b (32,) float64 of the fp32 operands -> Ref of the (B, h, w, 32) output."""
    mm = lambda a, m: torch.einsum("bchw,oc->bhwo", a, m.to(a.device))
    acc, A = mm(x, w), mm(x.abs(), w.abs())
    bb = b.to(x.device).view(1, 1, 1, -1)
    lead = (3.1 * 2.0 ** -18 + 770 * 2 * U32) if tensor_core else 256 * U32
    E = lead * A + U32 * (acc.abs() + bb.abs())
    ref = vr.Ref(acc + bb, E, out16=False)
    ref.A = A
    return ref


def simulate_feature_conv_tc(x, w, b, seed=0, drop_xl_wh=False):
    """CPU model of feature_conv1x1_tc_kernel: the three split products summed in fp32 in a shuffled order."""
    xh, xl = bf16_split(x)
    wh, wl = bf16_split(w)
    terms = [(xh, wh), (xh, wl)] + ([] if drop_xl_wh else [(xl, wh)])
    g = torch.Generator().manual_seed(seed)
    order = torch.randperm(len(terms), generator=g).tolist()
    perm = torch.randperm(x.shape[1], generator=g)
    acc = torch.zeros(x.shape[0], x.shape[2], x.shape[3], w.shape[0], dtype=torch.float32)
    for i in order:
        a, m = terms[i]
        acc = acc + torch.einsum("bchw,oc->bhwo", a[:, perm].float(), m[:, perm].float())
    return (acc + b.float()).to(F64)


# ---- bilinear sampling ------------------------------------------------------------------------------------------
def sample_coords(g, size):
    """The kernels' fp32 chain ix = fl(fl(fl(g + 1) / 2) * (size - 1)), in NumPy float32."""
    g = np.asarray(g, np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        return ((g + np.float32(1)) / np.float32(2)) * np.float32(size - 1)


def grid_for(ix, size):
    """fp32 grid values whose sample coordinate lies near ix (exactly ix where the chain allows it)."""
    return (2.0 * np.asarray(ix, np.float64) / (size - 1) - 1.0).astype(np.float32)


def bilinear_taps(ix, iy):
    """Four taps per point: integer coordinates (X, Y) and exact weights, from fp32 ix, iy (NumPy) as float64."""
    ix, iy = np.asarray(ix, np.float64), np.asarray(iy, np.float64)
    x0, y0 = np.floor(ix), np.floor(iy)
    wx1, wy1 = ix - x0, iy - y0
    wx0, wy0 = 1.0 - wx1, 1.0 - wy1
    big = np.float64(2 ** 40)                     # far outside any image: keeps the integer conversion defined
    x0, y0 = np.clip(x0, -big, big).astype(np.int64), np.clip(y0, -big, big).astype(np.int64)
    taps = []
    for t in range(4):
        X, Y = x0 + (t & 1), y0 + (t >> 1)
        wt = (wx1 if t & 1 else wx0) * (wy1 if t >> 1 else wy0)
        taps.append((X, Y, wt))
    return taps


def sample_ref(gather, taps, n_points):
    """gather(X, Y) -> (values (..., N, C) float64 with zeros where the tap is outside) for each tap; returns the Ref of
    the sampled values (..., N, C) and the per-point bound."""
    val = rad = None
    for X, Y, wt in taps:
        v = gather(X, Y)
        w = torch.from_numpy(wt).to(v.device).view(-1, 1)
        term, r = v * w, v.abs() * (8 * U32 * w.abs() + 3 * U32)
        val = term if val is None else val + term
        rad = r if rad is None else rad + r
    return vr.Ref(val, rad, out16=False)


def unproject_gather(feat, img_h, img_w):
    """Tap (X, Y) of the virtual img_h x img_w plane = pad(upsample_nearest(feat)): source cell (Y h / img_h,
    (X - pad) w / img_h), zero outside.  feat (B, h, w, C) float64.  gather.cells(X, Y) is the source cell index
    (-1 outside), the key the kernel merges taps by."""
    B, h, w, C = feat.shape
    pad = (img_w - img_h) // 2
    flat = feat.reshape(B, h * w, C)

    def cells(X, Y):
        xs = X - pad
        ok = (X >= 0) & (X < img_w) & (Y >= 0) & (Y < img_h) & (xs >= 0) & (xs < img_h)
        return np.where(ok, (np.clip(Y, 0, img_h - 1) * h) // img_h * w + (np.clip(xs, 0, img_h - 1) * w) // img_h, -1)

    def gather(X, Y):
        cell = cells(X, Y)
        idx = torch.from_numpy(np.maximum(cell, 0)).to(feat.device)
        return flat[:, idx] * torch.from_numpy(cell >= 0).to(feat.device).view(1, -1, 1)
    gather.cells = cells
    return gather


def image_gather(img):
    """Tap (X, Y) of an NCHW image, zero outside; returns (B, N, C)."""
    B, C, H, W = img.shape
    flat = img.reshape(B, C, H * W)

    def gather(X, Y):
        ok = (X >= 0) & (X < W) & (Y >= 0) & (Y < H)
        idx = torch.from_numpy(np.where(ok, np.clip(Y, 0, H - 1) * W + np.clip(X, 0, W - 1), 0)).to(img.device)
        return flat[:, :, idx].transpose(1, 2) * torch.from_numpy(ok).to(img.device).view(1, -1, 1)
    return gather


def simulate_sample_f32(gather, ix, iy, order=(0, 1, 2, 3), drop_tap=None):
    """CPU model of unproject_kernel: fp32 weights, taps that share a source cell merged in fp32 (gather.cells), the
    surviving taps accumulated in `order` with one rounding per fmaf.  drop_tap: that tap's weight is lost before the
    merge."""
    ix32, iy32 = np.asarray(ix, np.float32), np.asarray(iy, np.float32)
    with np.errstate(invalid="ignore"):
        x0, y0 = np.floor(ix32), np.floor(iy32)
        wx1, wy1 = ix32 - x0, iy32 - y0
        wx0, wy0 = (x0 + np.float32(1)) - ix32, (y0 + np.float32(1)) - iy32
    taps = bilinear_taps(ix, iy)
    wt = [((wx1 if t & 1 else wx0) * (wy1 if t >> 1 else wy0)).astype(np.float32) for t in range(4)]
    if drop_tap is not None:
        wt[drop_tap] = np.zeros_like(wt[drop_tap])
    cell = [gather.cells(X, Y) for X, Y, _ in taps]
    for t in range(1, 4):
        for u in range(t):
            same = (cell[t] >= 0) & (cell[t] == cell[u])
            wt[u] = np.where(same, wt[u] + wt[t], wt[u]).astype(np.float32)
            cell[t] = np.where(same, -1, cell[t])
    acc = None
    for t in order:
        X, Y, _ = taps[t]
        v = gather(X, Y)
        w = torch.from_numpy(np.where(cell[t] >= 0, wt[t], 0).astype(np.float64)).to(v.device).view(-1, 1)
        step = v * w if acc is None else v * w + acc
        acc = step.to(torch.float32).to(F64)
    return acc


# ---- soft-argmax ------------------------------------------------------------------------------------------------
def softargmax_launch(BJ, N, sms=148):
    """(splits, chunk) of sa_splits in csrc/softargmax.cu."""
    splits = min(max((48 * sms + BJ - 1) // BJ, 1), 64)
    unit = 256 * 16
    chunk = ((N + splits - 1) // splits + unit - 1) // unit * unit
    return (N + chunk - 1) // chunk, chunk


def softargmax_ref(x, mult, softmax, coords):
    """x (B, J, N) float64 of the fp32 logits, coords (N, 3) float64 of the fp32 coordinates.  Returns (kp Ref
    (B, J, 3), volume Ref (B, J, N))."""
    B, J, N = x.shape
    mult = float(np.float32(mult))                        # the kernel takes the multiplier as an fp32 argument
    splits, chunk = softargmax_launch(B * J, N)
    iters = chunk // 4096
    Ka, Km = 4 * iters + 13 + splits, iters + 13 + splits
    y = x * mult
    fin = torch.isfinite(y)
    c = coords.to(x.device)
    if not softmax:
        w = y.clamp_min(0).to(torch.float32).to(F64)
        kp = torch.einsum("bjn,nk->bjk", y.clamp_min(0), c)
        E = (Ka + 1) * U32 * torch.einsum("bjn,nk->bjk", w, c.abs())
        return vr.Ref(kp, E, out16=False), vr.Ref(w, torch.zeros_like(w), out16=False)
    M = torch.where(fin, y, torch.full_like(y, -math.inf)).amax(dim=2, keepdim=True)
    lo = torch.where(fin, y, torch.full_like(y, math.inf)).amin(dim=2, keepdim=True)
    D = M - lo
    d = y - M
    e = torch.exp(d)
    s = e.sum(dim=2, keepdim=True)
    p = e / s
    delta = torch.where(fin, 1.01 * U32 * (y.abs() + 3 * d.abs()) + 2.0 ** -22, torch.zeros_like(y))
    path = Ka * U32 + Km * U32 * (5 + 3 * D)
    rel_s = (p * delta).sum(dim=2, keepdim=True) + path
    vol_E = 1.01 * p * (delta + rel_s + 2.0 ** -23) + 2.0 ** -147
    kp = torch.einsum("bjn,nk->bjk", p, c)
    kp_E = 1.01 * (torch.einsum("bjn,nk->bjk", p * (delta + path), c.abs()) + kp.abs() * (rel_s + 2.0 ** -22))
    return vr.Ref(kp, kp_E, out16=False), vr.Ref(p, vol_E, out16=False)


# ---- comparisons ------------------------------------------------------------------------------------------------
def err_ratio(got, ref):
    """Largest |got - ref| / bound (for the report)."""
    r = (got.to(F64) - ref.value).abs() / (ref.radius + 2.0 ** -149)
    return float(r.max())


def assert_within_flat(got, ref, where, limit=8):
    """assert_within for tensors of any shape: the first wrong elements and their count."""
    bad = ~vr.within_mask(got, ref)
    if bool(bad.any()):
        idx = bad.nonzero()
        g = got.to(F64)
        lines = [f"{where}: {idx.shape[0]} of {bad.numel()} elements outside the bound"]
        for row in idx[:limit].tolist():
            t = tuple(row)
            lines.append(f"  {t}: got {g[t].item()!r}, want {ref.value[t].item()!r} +- {ref.radius[t].item():.3e}")
        raise AssertionError("\n".join(lines))


def assert_equal_flat(got, want, where, limit=8):
    g, w = got.to(F64), want.to(F64)
    bad = ~(g == w)
    if bool(bad.any()):
        idx = bad.nonzero()
        lines = [f"{where}: {idx.shape[0]} of {bad.numel()} elements differ"]
        for row in idx[:limit].tolist():
            t = tuple(row)
            lines.append(f"  {t}: got {g[t].item()!r}, want {w[t].item()!r}")
        raise AssertionError("\n".join(lines))


# ---- fisheye projection (csrc/geometry.cu project_voxel) ----------------------------------------------------------------
ATANF_ULP = 2         # atanf: 2 ulp over the full range (CUDA 12.9 Math API, single-precision functions table)
TAU32 = 2.0 ** -150   # absolute rounding error of an fp32 result in the subnormal range


def _ulp32(x):
    """ulp of an fp32 value of magnitude <= |x| + ... (normal range; 2^-149 below it)."""
    e = np.floor(np.log2(np.maximum(np.abs(x), 2.0 ** -126)))
    return np.exp2(e - 23)


def w2c_coeffs(calib):
    """The kernel's fp32 copies of the W2C polynomial and the centre, as float64 values."""
    a = np.asarray(calib["w2c"], np.float64).astype(np.float32).astype(np.float64)
    cx, cy = (np.float64(np.float32(v)) for v in calib["center"])
    return a, cx, cy


def project_ref(pts, calib):
    """Float64 value of the Scaramuzza expression at fp32 points (N, 3), with a running error bound of the fp32
    evaluation (u = 2^-24 per rounded op plus 2^-150 absolute for subnormal results, sqrtf correctly rounded, atanf
    ATANF_ULP ulp; input errors propagated through each op's derivative).  Returns (px (N, 2), radius (N, 2), theta,
    r2_32), r2_32 being the fp32 value of X^2 + Y^2 (0 where the kernel takes its r == 0 branch)."""
    a, cx, cy = w2c_coeffs(calib)
    p = np.asarray(pts, np.float32).astype(np.float64)
    X, Y, z = p[:, 0], p[:, 1], -p[:, 2]
    rnd = lambda v, e: U32 * (np.abs(v) + e) + TAU32         # rounding of a result v known to within e
    X2, Y2 = X * X, Y * Y
    eX2, eY2 = rnd(X2, 0), rnd(Y2, 0)
    s = X2 + Y2
    es = eX2 + eY2
    es = es + rnd(s, es)
    r = np.sqrt(s)
    er = es / (r + np.sqrt(np.maximum(s - es, 0.0)))
    er = er + rnd(r, er)
    with np.errstate(divide="ignore", invalid="ignore"):
        lo = np.maximum(r - er, 0.0)
        q = z / r
        eq = np.abs(z) * er / (r * lo)
        eq = eq + rnd(q, eq)
        th = np.arctan(q)
        qlo = np.maximum(np.abs(q) - eq, 0.0)
        eth = eq / (1.0 + qlo * qlo)
        eth = eth + ATANF_ULP * _ulp32(np.abs(th) + eth)
        inv = 1.0 / r
        einv = er / (r * lo)
        einv = einv + rnd(inv, einv)
        t, et = np.ones_like(th), np.zeros_like(th)
        rho, erho = np.full_like(th, a[0]), np.zeros_like(th)
        for i in range(1, 11):
            tn = t * th
            etn = np.abs(t) * eth + np.abs(th) * et + et * eth
            t, et = tn, etn + rnd(tn, etn)
            m = t * a[i]
            em = abs(a[i]) * et
            em = em + rnd(m, em)
            rho = rho + m
            erho = erho + em
            erho = erho + rnd(rho, erho)
        out, rad = [], []
        for V, c0 in ((X, cx), (Y, cy)):
            xi = V * inv
            exi = np.abs(V) * einv
            exi = exi + rnd(xi, exi)
            pm = xi * rho
            epm = np.abs(xi) * erho + np.abs(rho) * exi + exi * erho
            epm = epm + rnd(pm, epm)
            px = pm + c0
            epx = epm + rnd(px, epm)
            out.append(px)
            rad.append(1.001 * epx + 2.0 ** -40 * np.abs(px))   # the float64 evaluation itself
    x32, y32 = p[:, 0].astype(np.float32), p[:, 1].astype(np.float32)
    with np.errstate(over="ignore", under="ignore"):
        r2_32 = (x32 * x32 + y32 * y32).astype(np.float64)
    return np.stack(out, 1), np.stack(rad, 1), th, r2_32


def normalise_ref(px, rad, hm_h, hm_w):
    """g = 2 (p / [W, H] - 0.5) in fp32 (division, subtraction, exact doubling) around the projection's bound."""
    out, orad = [], []
    for k, size in ((0, hm_w), (1, hm_h)):
        d = px[:, k] / size
        ed = rad[:, k] / size
        ed = ed + U32 * (np.abs(d) + ed) + TAU32
        s = d - 0.5
        es = ed + U32 * (np.abs(s) + ed) + TAU32
        out.append(2 * s)
        orad.append(2 * es)
    return np.stack(out, 1), np.stack(orad, 1)


def simulate_project_f32(pts, calib, atan_ulps=0, seed=0, drop=None, swap_centre=False, no_flip=False):
    """The kernel in NumPy float32: atan perturbed by up to `atan_ulps` ulp (random direction per point); planted
    defects: drop=i leaves out coefficient a_i, swap_centre exchanges cx and cy, no_flip takes theta from +Z."""
    a, cx, cy = w2c_coeffs(calib)
    a = a.astype(np.float32)
    if swap_centre:
        cx, cy = cy, cx
    cx, cy = np.float32(cx), np.float32(cy)
    p = np.asarray(pts, np.float32)
    X, Y = p[:, 0], p[:, 1]
    z = p[:, 2] if no_flip else p[:, 2] * np.float32(-1)
    with np.errstate(all="ignore"):
        r = np.sqrt(X * X + Y * Y)
        th = np.arctan(z / r).astype(np.float32)
        if atan_ulps:
            rng = np.random.default_rng(seed)
            k = rng.integers(-atan_ulps, atan_ulps + 1, th.shape)
            for _ in range(atan_ulps):
                th = np.where(k > 0, np.nextafter(th, np.float32(np.inf)), np.where(k < 0, np.nextafter(th, np.float32(-np.inf)), th))
                k = k - np.sign(k)
        inv = np.float32(1) / r
        rho = np.full_like(th, a[0])
        t = np.ones_like(th)
        for i in range(1, 11):
            t = t * th
            if i != drop:
                rho = rho + t * a[i]
        px = (X * inv) * rho + cx
        py = (Y * inv) * rho + cy
    return np.stack([px, py], 1).astype(np.float64)


def w2c_within(got, ref, rad):
    got = np.asarray(got, np.float64)
    return np.isfinite(got) & (np.abs(got - ref) <= rad)

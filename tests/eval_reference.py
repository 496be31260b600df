"""Float64 reference of the pose-error kernel (csrc/eval.cu) with a per-frame bound, and a NumPy model of the kernel.

The reference is oracle.umeyama / align_skeleton restated for a batch (np.linalg.svd per frame).  The bound of one
frame follows from the conditioning of its cross-covariance C = A^T G / J (A, G the centred poses, eps = 2^-53):

- the kernel's centred coordinates are off by at most dA = (J + 4) eps max|P| (dG alike: the mean is a J-term sum);
- its C (fp64, FMA-contracted, another summation order) by
    dC = ((J + 4) eps |A|_F |G|_F + sqrt(3 J) (dA |G|_F + dG |A|_F)) / J        (Frobenius);
- the rotation is the polar factor of C, whose sensitivity is 1 / (S1 + S2) (S2 signed as in umeyama):
    dR = 4 dC / (S1 + S2) + 4 eps                                              (every entry);
  when S1 + S2 <= 1e4 dC the rotation is not unique (rank C <= 1 up to rounding) and nothing that depends on it is
  compared with the oracle; such a frame is checked for |R^T R - I| <= 1e-12, det R = +1, optimality
  (trace(R^T C) = S0 + S1 + S2), its sum of squared residuals (unique) and c, t, aligned against its own transform;
- trace(R^T C) is stationary in R:  dTr = 4 sqrt(3) dC + 3 S0 dR^2 + 16 eps (S0 + S1 + |S2|);
- varp:  dV = 2 (J + 4) eps varp + 2 sqrt(3 J) dA |A|_F / J;  c = tr / varp:  dc = 1.01 (dTr + |c| dV) / varp + 4 eps |c|;
- t = mQ - c mP R, aligned = cs P R + t and PA-MPJPE by first-order propagation with 4 eps per rounded operation;
- MPJPE: (J + 8) eps MPJPE.
"""
import numpy as np

EPS = 2.0 ** -53
FREE = 1e4                       # S1 + S2 <= FREE dC: the rotation is not unique


def oracle(pred, gt, scale):
    """orc.align_skeleton / umeyama per frame, batched: dict of mpjpe (B,), pampjpe (B,), aligned (B,J,3),
    gt_out (B,J,3), c (B,), R (B,3,3), t (B,3), S (B,3) signed, C (B,3,3), A and G (centred poses), varp (B,)."""
    P = np.array(pred, dtype=np.float64)
    Q = np.array(gt, dtype=np.float64)
    J = P.shape[1]
    mpjpe = np.linalg.norm(P - Q, axis=2).mean(1)
    if not scale:
        P -= P.mean(1, keepdims=True)
        Q -= Q.mean(1, keepdims=True)
    mP, mQ = P.mean(1), Q.mean(1)
    A, G = P - mP[:, None], Q - mQ[:, None]
    C = np.einsum("bji,bjk->bik", A, G) / J
    V, S, W = np.linalg.svd(C)
    flip = np.linalg.det(V) * np.linalg.det(W) < 0.0
    S[flip, 2] *= -1
    V[flip, :, 2] *= -1
    R = V @ W
    varp = np.var(P, axis=1).sum(1)
    with np.errstate(divide="ignore", invalid="ignore"):
        c = 1 / varp * S.sum(1)
        t = mQ - np.einsum("bi,bik->bk", mP, c[:, None, None] * R)
        PR = np.einsum("bji,bik->bjk", P, R)
        aligned = (PR * c[:, None, None] if scale else PR) + t[:, None]
    pampjpe = np.linalg.norm(aligned - Q, axis=2).mean(1)
    return dict(mpjpe=mpjpe, pampjpe=pampjpe, aligned=aligned, gt_out=Q, c=c, R=R, t=t, S=S, C=C, A=A, G=G, P=P,
                mP=mP, mQ=mQ, varp=varp, scale=scale, raw_P=np.asarray(pred, np.float64), raw_Q=np.asarray(gt, np.float64))


def bounds(ref):
    """Per-frame radii for the outputs of `oracle` (same keys), and the mask of frames whose rotation is free."""
    P, A, G, S = ref["P"], ref["A"], ref["G"], ref["S"]
    J = P.shape[1]
    r3J = np.sqrt(3.0 * J)
    mabsP = np.abs(ref["raw_P"]).max((1, 2))
    mabsQ = np.abs(ref["raw_Q"]).max((1, 2))
    dA, dG = (J + 4) * EPS * mabsP, (J + 4) * EPS * mabsQ
    dmP, dmQ = (J + 1) * EPS * mabsP, (J + 1) * EPS * mabsQ
    nA, nG = np.linalg.norm(A, axis=(1, 2)), np.linalg.norm(G, axis=(1, 2))
    dC = ((J + 4) * EPS * nA * nG + r3J * (dA * nG + dG * nA)) / J
    s12 = S[:, 1] + S[:, 2]
    free = ~(s12 > FREE * dC)
    with np.errstate(divide="ignore", invalid="ignore"):
        dR = np.where(free, np.nan, 4 * dC / s12 + 4 * EPS)
        dRz = np.where(free, 0.0, dR)                      # free frames: the terms of their own rotation only
        S_abs = np.abs(S).sum(1)
        dTr = 4 * np.sqrt(3) * dC + 3 * S[:, 0] * dRz ** 2 + 16 * EPS * S_abs
        varp = ref["varp"]
        c = ref["c"]
        dV = 2 * (J + 4) * EPS * varp + 2 * r3J * dA * nA / J
        dc = 1.01 * (dTr + np.abs(c) * dV) / varp + 4 * EPS * np.abs(c)
        mP, mQ = ref["mP"], ref["mQ"]
        smP = np.abs(mP).sum(1)
        t_rnd = 4 * EPS * (np.abs(mQ).max(1) + np.abs(c) * smP)
        dt = dmQ + dc * smP + np.abs(c) * dmP * 3 + t_rnd
        dt_rot = np.abs(c) * smP * dRz                     # the part of dt owed to dR
        cs = c if ref["scale"] else np.ones_like(c)
        dcs = dc if ref["scale"] else np.zeros_like(c)
        absP = np.abs(P).sum(2)                            # (B, J): sum_i |P_ji|
        da = np.zeros_like(dA) if ref["scale"] else 3 * dA    # scale=False: the kernel centres pred itself
        dal = (dcs[:, None] * absP + np.abs(cs)[:, None] * (absP * dRz[:, None] + da[:, None]) + (dt + dt_rot)[:, None]
               + 4 * EPS * (np.abs(cs)[:, None] * absP + np.abs(ref["t"]).max(1)[:, None]))
        dg = np.zeros_like(dA) if ref["scale"] else EPS * np.abs(ref["gt_out"]).max((1, 2)) + 2 * dmQ
        dpa = np.sqrt(3) * (dal + dg[:, None]).mean(1) + (J + 8) * EPS * ref["pampjpe"]
    return dict(free=free, dC=dC, dR=dR, dTr=dTr, dc=dc, dt=dt + dt_rot, aligned=dal, gt_out=dg,
                pampjpe=dpa, mpjpe=(J + 8) * EPS * ref["mpjpe"], dV=dV, dA=dA, dG=dG, nA=nA, nG=nG)


def _bad(got, want, radius):
    """Mask of elements outside [want - radius, want + radius]; NaN in want demands NaN in got."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    nan_want = np.isnan(want)
    ok = np.where(nan_want, np.isnan(got), np.isfinite(got) & (np.abs(got - want) <= radius))
    return ~ok


def check(out, ref, bnd, where, frames=None):
    """Compare kernel outputs (dict of mpjpe, pampjpe, aligned, gt_out, transform (B,13)) with the reference.
    Returns the largest |err| / bound per quantity over the frames with a unique rotation.  Raises on a violation."""
    B = ref["c"].shape[0]
    sel = np.ones(B, bool) if frames is None else frames
    free = bnd["free"] & sel
    uniq = ~bnd["free"] & sel
    T = out["transform"]
    c_k, R_k, t_k = T[:, 0], T[:, 1:10].reshape(-1, 3, 3), T[:, 10:13]
    errs, fails = {}, []

    def cmp(name, got, want, radius, mask):
        if not mask.any():
            return
        g, w = np.asarray(got)[mask], np.asarray(want)[mask]
        r = np.broadcast_to(np.asarray(radius, np.float64), np.asarray(want).shape)[mask]
        bad = _bad(g, w, r)
        if bad.any():
            i = np.argwhere(bad)[0]
            frame = np.flatnonzero(mask)[i[0]]
            fails.append(f"{where}: {name}: {int(bad.sum())} of {bad.size} elements outside the bound; first at frame "
                         f"{frame} {tuple(i[1:])}: got {g[tuple(i)]!r}, want {w[tuple(i)]!r} +- {r[tuple(i)]:.3e}")
        fin = np.isfinite(w) & np.isfinite(g) & (r > 0)
        if fin.any():
            errs[name] = max(errs.get(name, 0.0), float((np.abs(g - w)[fin] / r[fin]).max()))

    all_ = sel
    cmp("mpjpe", out["mpjpe"], ref["mpjpe"], bnd["mpjpe"], all_)
    cmp("gt_out", out["gt_out"], ref["gt_out"], bnd["gt_out"][:, None, None], all_)
    cmp("c", c_k, ref["c"], bnd["dc"], all_)
    cmp("R", R_k, ref["R"], bnd["dR"][:, None, None], uniq)
    cmp("t", t_k, ref["t"], bnd["dt"][:, None], uniq)
    cmp("aligned", out["aligned"], ref["aligned"], bnd["aligned"][..., None], uniq)
    cmp("pampjpe", out["pampjpe"], ref["pampjpe"], bnd["pampjpe"], uniq)
    # every frame: R is a rotation, optimal for the oracle's C, and c, t, aligned follow from the frame's own transform
    fin = all_ & np.isfinite(R_k).all((1, 2))
    I = np.eye(3)
    cmp("R^T R - I", np.einsum("bki,bkj->bij", R_k, R_k) - I, np.zeros((B, 3, 3)), 1e-12, fin)
    cmp("det R", np.linalg.det(np.where(fin[:, None, None], R_k, I)), np.ones(B), 1e-12, fin)
    tr = np.einsum("bik,bik->b", R_k, ref["C"])
    cmp("trace(R^T C)", tr, ref["S"].sum(1), bnd["dTr"], all_)
    with np.errstate(invalid="ignore"):
        t_own = ref["mQ"] - np.einsum("bi,bik->bk", ref["mP"], c_k[:, None, None] * R_k)
        cmp("t (own R)", t_k, t_own, bnd["dt"][:, None], free)
        cs = c_k if ref["scale"] else np.ones_like(c_k)
        al_own = np.einsum("bji,bik->bjk", ref["P"], R_k) * cs[:, None, None] + t_k[:, None]
        cmp("aligned (own transform)", out["aligned"], al_own, bnd["aligned"][..., None], free)
        ssr_k = ((out["aligned"] - out["gt_out"]) ** 2).sum((1, 2))
        ssr_o = ((ref["aligned"] - ref["gt_out"]) ** 2).sum((1, 2))
        cmp("sum of squared residuals", ssr_k, ssr_o, ssr_bound(ref, bnd), free)
        cmp("pampjpe (own transform)", out["pampjpe"], np.linalg.norm(out["aligned"] - out["gt_out"], axis=2).mean(1),
            (ref["P"].shape[1] + 8) * EPS * np.abs(out["pampjpe"]) + 1e-300, free)
    if fails:
        raise AssertionError("\n".join(fails))
    return errs


def ssr_bound(ref, bnd):
    """The optimal sum of squared residuals is J (varq - tr^2 / varp) (scale) or J (varp + varq - 2 tr): its error
    follows from dTr and dV, plus the rounding of the residuals themselves (their radius E without the dR terms)."""
    J = ref["P"].shape[1]
    tr = np.abs(ref["S"].sum(1))
    varp = ref["varp"]
    nG = bnd["nG"]
    if ref["scale"]:
        d = J * (2 * tr * bnd["dTr"] / varp + tr ** 2 * bnd["dV"] / varp ** 2) + 2 * bnd["dG"] * nG * np.sqrt(3 * J)
    else:
        d = 2 * J * bnd["dTr"] + J * bnd["dV"] + 2 * np.sqrt(3 * J) * bnd["dG"] * nG
    ssr = ((ref["aligned"] - ref["gt_out"]) ** 2).sum((1, 2))
    E = np.sqrt(3 * J) * (bnd["aligned"].max(1) + bnd["gt_out"])
    return d + 2 * np.sqrt(ssr) * E + E ** 2 + 8 * J * EPS * ssr


# ---- a NumPy model of the kernel (float64, scalar, no FMA) -------------------------------------------------------
def _jacobi(a):
    a, e = a.copy(), np.eye(3)
    with np.errstate(over="ignore"):                      # theta^2 may overflow, as in the kernel: then t = 0
        return _jacobi_sweeps(a, e)


def _jacobi_sweeps(a, e):
    for _ in range(30):
        off = a[0, 1] ** 2 + a[0, 2] ** 2 + a[1, 2] ** 2
        if off <= 1e-60 * (a[0, 0] ** 2 + a[1, 1] ** 2 + a[2, 2] ** 2) or off == 0.0:
            break
        for p, q in ((0, 1), (0, 2), (1, 2)):
            if a[p, q] == 0.0:
                continue
            th = (a[q, q] - a[p, p]) / (2.0 * a[p, q])
            t = (1.0 if th >= 0.0 else -1.0) / (abs(th) + np.sqrt(th * th + 1.0))
            c = 1.0 / np.sqrt(t * t + 1.0)
            s = t * c
            J = np.eye(3)
            J[p, p], J[p, q], J[q, p], J[q, q] = c, s, -s, c
            a = J.T @ a @ J
            e = J.T @ e
    w = np.diag(a).copy()
    o = np.argsort(-w, kind="stable")
    return w[o], e[o]


def model_frame(P, Q, scale, reverse=False, legacy_v=False, flip_r2=False):
    """One frame of the kernel: returns (mpjpe, pampjpe, aligned, gt_out, transform).  reverse: sum the joints in the
    other order; legacy_v: the V construction before the orthonormal completion; flip_r2: negate R's third column."""
    P, Q = np.asarray(P, np.float64), np.asarray(Q, np.float64)
    J = P.shape[0]
    order = range(J - 1, -1, -1) if reverse else range(J)
    mp, mq, dist = np.zeros(3), np.zeros(3), 0.0
    for j in order:
        dist += np.sqrt(((P[j] - Q[j]) ** 2).sum())
        mp, mq = mp + P[j], mq + Q[j]
    mp, mq = mp / J, mq / J
    offp, offq = (np.zeros(3), np.zeros(3)) if scale else (mp, mq)
    cp, cq = mp - offp, mq - offq
    C, varp = np.zeros((3, 3)), 0.0
    for j in order:
        a, q = (P[j] - offp) - cp, (Q[j] - offq) - cq
        varp += (a * a).sum()
        C += np.outer(a, q)
    C, varp = C / J, varp / J
    ev, W = _jacobi(C.T @ C)
    S = np.sqrt(np.maximum(ev, 0.0))
    tiny = 1e-14 * (S[0] if S[0] > 0 else 1.0)
    U = np.array([C @ W[c] for c in range(3)])
    V = np.eye(3)
    if legacy_v:
        for c in range(3):
            if S[c] > tiny:
                V[:, c] = U[c] / S[c]
            elif c == 2:
                V[:, 2] = np.cross(V[:, 0], V[:, 1])
            else:
                V[:, c] = np.eye(3)[c]
    else:
        n0 = np.linalg.norm(U[0])
        if S[0] > tiny and n0 > 0:
            v0 = U[0] / n0
            v1 = U[1] - (v0 @ U[1]) * v0
            n1 = np.linalg.norm(v1)
            if not (S[1] > tiny and n1 > tiny):
                v1 = np.cross(v0, np.eye(3)[int(np.argmin(np.abs(v0)))])
                n1 = np.linalg.norm(v1)
            V = np.stack([v0, v1 / n1, np.cross(v0, v1 / n1)], 1)
        S = np.array([V[:, c] @ U[c] for c in range(3)])
    if np.linalg.det(V) * np.linalg.det(W) < 0.0:
        S[2], V[:, 2] = -S[2], -V[:, 2]
    R = V @ W
    if flip_r2:
        R[:, 2] = -R[:, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        c = S.sum() / varp
        t = cq - c * (cp @ R)
        cs = c if scale else 1.0
        aligned = cs * ((P - offp) @ R) + t
    gt_out = Q - offq
    pa = np.linalg.norm(aligned - gt_out, axis=1)
    pa = sum(pa[j] for j in order) / J
    return dist / J, pa, aligned, gt_out, np.concatenate([[c], R.reshape(-1), t])


def model(pred, gt, scale, **kw):
    outs = [model_frame(p, g, scale, **kw) for p, g in zip(pred, gt)]
    return dict(mpjpe=np.array([o[0] for o in outs]), pampjpe=np.array([o[1] for o in outs]),
                aligned=np.stack([o[2] for o in outs]), gt_out=np.stack([o[3] for o in outs]),
                transform=np.stack([o[4] for o in outs]))


# ---- cases ---------------------------------------------------------------------------------------------------------
def _rot(rng, n):
    q = rng.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                     2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                     2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], 1).reshape(n, 3, 3)


def make_case(kind, B, J, seed):
    """(pred, gt) float64 (B, J, 3) of one kind of frame."""
    rng = np.random.default_rng(seed)
    gt = rng.normal(0, 0.5, (B, J, 3)) + rng.normal(0, 1, (B, 1, 3))
    noise = rng.normal(0, 0.05, (B, J, 3))
    rot = _rot(rng, B)
    if kind == "generic":
        pred = np.einsum("bji,bik->bjk", gt, rot) * rng.uniform(0.8, 1.2, (B, 1, 1)) + noise
    elif kind == "reflected":
        pred = gt * np.array([1.0, 1.0, -1.0]) + noise                      # det C < 0
    elif kind == "planar":
        gt[:, :, 2] = 0.25                                                  # exactly planar
        pred = gt + noise
    elif kind.startswith("near-planar-"):
        r = float(kind.split("-")[-1])
        base = rng.normal(0, 0.5, (B, J, 3))
        base[:, :, 2] *= r
        gt = np.einsum("bji,bik->bjk", base, rot) + 0.3
        pred = gt + noise
    elif kind == "collinear-gt":
        gt = rng.normal(0, 0.5, (B, J, 1)) * rng.normal(0, 1, (B, 1, 3)) + rng.normal(0, 1, (B, 1, 3))
        pred = gt + noise
    elif kind == "collinear-pred":
        s = rng.integers(-64, 65, (B, J, 1)) / 64.0                        # exact in float32 too
        pred = s * np.array([1.0, 2.0, 2.0]) + np.array([0.5, -0.25, 1.0])
    elif kind == "pred-constant":
        pred = np.broadcast_to(rng.integers(-8, 9, (B, 1, 3)) / 8.0, (B, J, 3)).copy()
    elif kind == "gt-constant":
        gt = np.broadcast_to(rng.normal(0, 1, (B, 1, 3)), (B, J, 3)).copy()
        pred = gt + noise
    elif kind == "equal":
        gt = gt.astype(np.float32).astype(np.float64)
        pred = gt.copy()
    elif kind == "isotropic":                                               # C = s I-like: Jacobi exits at once
        assert J == 6
        octa = np.concatenate([np.eye(3), -np.eye(3)]) * 0.5
        gt = np.broadcast_to(octa, (B, J, 3)).copy()
        pred = gt[:, :, [1, 2, 0]].copy()                                    # an exact rotation (axis permutation)
    elif kind == "translated":
        gt = rng.normal(0, 0.5, (B, J, 3)) + 1e3
        pred = gt + rng.normal(0, 1e-3, (B, J, 3))
    else:
        raise ValueError(kind)
    return pred, gt

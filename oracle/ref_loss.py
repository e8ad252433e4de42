"""Oracle (test infrastructure, not product): thermal-aware training loss.

Restates /root/reference/utils/loss.py.  Two independent forms:

* ``*_torch``  fp32 torch-CPU graph (autograd gives the reference gradients);
  op order follows the reference where rounding could matter.
* ``loss_fwd_bwd_f64``  numpy float64 closed form of forward AND backward
  (SURVEY.md Appendix A) -- the "true value" both the CUDA kernels and the
  fp32 reference are compared with when the tolerance is tight.

Pinned against the unmodified reference by tests/test_oracle_pin.py (live,
build container only) and tests/golden/loss_*.npz (travels to the GPU box).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

# constants hard-coded in the reference
EPS = 1e-5            # utils/loss.py:240
THERMAL_FACTOR = 8.0  # utils/loss.py:252
CLAMP_VIEW = (0.4, 0.5)  # utils/loss.py:253-256 (view 1, view 2)
HUBER_DELTA = 0.1     # utils/loss.py:267
CONF_MIN, CONF_MAX = 1e-5, 10.0  # utils/loss.py:91-92
GRAY = (0.299, 0.587, 0.114)     # utils/loss.py:120


# --------------------------------------------------------------------------- torch fp32
def confidence_weighted_regression_loss_torch(p1, p2, g1, g2, c1=None, c2=None, alpha=0.2):
    """utils/loss.py:75-98."""
    total = 0
    for p, g, c in ((p1, g1, c1), (p2, g2, c2)):
        l = (p - g).abs().mean(dim=-1)                       # :82-83
        if c is None:
            c = torch.ones_like(l)                           # :86-89
        c = c.clamp(min=CONF_MIN, max=CONF_MAX)              # :91-92
        total = total + (c * l - alpha * torch.log(c)).mean()  # :95-96
    return total


def plain_confidence_loss_torch(p1, p2, g1, g2, conf1, conf2, alpha=0.2):
    """train_thermal_dustr.py:278-279,305-318 ("original loss calculation", --use_thermal_aware_loss off): the
    confidence is clamped from below only (clamp(min=1e-5)); no upper clamp at 10 as in utils/loss.py:91-92."""
    conf1, conf2 = torch.clamp(conf1, min=1e-5), torch.clamp(conf2, min=1e-5)        # :278-279
    loss1 = torch.abs(p1 - g1).mean(dim=-1)                                          # :307
    loss2 = torch.abs(p2 - g2).mean(dim=-1)                                          # :308
    w1 = (conf1 * loss1 - alpha * torch.log(conf1)).mean()                           # :313
    w2 = (conf2 * loss2 - alpha * torch.log(conf2)).mean()                           # :314
    return w1 + w2                                                                   # :317


def _gray_torch(t):
    """utils/loss.py:119-124 (left-to-right fp32 sum)."""
    if t.shape[0] == 3:
        return GRAY[0] * t[0] + GRAY[1] * t[1] + GRAY[2] * t[2]
    return t[0]


def _padded_absdiff_torch(a):
    """Zero-padded forward |differences|, utils/loss.py:184-237."""
    dx = torch.zeros_like(a)
    dy = torch.zeros_like(a)
    if a.shape[1] > 1:
        dx[:, :-1] = (a[:, 1:] - a[:, :-1]).abs()
    if a.shape[0] > 1:
        dy[:-1, :] = (a[1:, :] - a[:-1, :]).abs()
    return dx, dy


def _pool_torch(a, s):
    """utils/loss.py:159-174."""
    return F.avg_pool2d(a[None, None], s, s).squeeze()


def _huber_torch(d):
    """utils/loss.py:275-285 (strict <)."""
    return torch.where(d < HUBER_DELTA, 0.5 * d.pow(2), HUBER_DELTA * (d - 0.5 * HUBER_DELTA))


def enhanced_thermal_aware_loss_torch(pred_pts1, pred_pts2, gt_pts1, gt_pts2,
                                      confidences1=None, confidences2=None,
                                      thermal_img1=None, thermal_img2=None,
                                      alpha=0.2, edge_weight=0.5, smoothness_weight=0.3,
                                      detail_weight=0.3, multi_scale=True):
    """utils/loss.py:100-305.  Returns (total, dict of python floats)."""
    p1, p2, g1, g2, c1, c2, t1, t2 = (pred_pts1, pred_pts2, gt_pts1, gt_pts2, confidences1,
                                      confidences2, thermal_img1, thermal_img2)
    basic = confidence_weighted_regression_loss_torch(p1, p2, g1, g2, c1, c2, alpha)
    edge = smooth = detail = 0
    if t1 is not None and t2 is not None:
        if not (isinstance(t1, torch.Tensor) and t1.dim() == 3):
            # reference: thermal_gray1 unbound -> NameError (utils/loss.py:118-140)
            raise NameError("thermal_gray1")
        for s in ([1, 2] if multi_scale else [1]):          # :133
            lam = 1.0 if s == 1 else 0.7 / s                 # :288
            for view, (p, g, t) in enumerate(((p1, g1, t1), (p2, g2, t2))):
                gr, z, gz = _gray_torch(t), p[..., 2], g[..., 2]
                if s > 1:
                    gr, z, gz = _pool_torch(gr, s), _pool_torch(z, s), _pool_torch(gz, s)
                tx, ty = _padded_absdiff_torch(gr)
                ax, ay = _padded_absdiff_torch(z)
                bx, by = _padded_absdiff_torch(gz)
                nx = tx / (tx.mean() + EPS)                  # :240-249
                ny = ty / (ty.mean() + EPS)
                m = CLAMP_VIEW[view]
                w = torch.exp(-nx.clamp(0, m) * THERMAL_FACTOR) * \
                    torch.exp(-ny.clamp(0, m) * THERMAL_FACTOR)  # :253-256
                e = (ax * (1 - w)).mean() + (ay * (1 - w)).mean()        # :259-260
                sm = (ax.pow(2) * w).mean() + (ay.pow(2) * w).mean()     # :263-264
                d = _huber_torch((ax - bx).abs()).mean() + _huber_torch((ay - by).abs()).mean()
                edge = edge + lam * e
                smooth = smooth + lam * sm
                detail = detail + lam * d
    total = basic + edge_weight * edge + smoothness_weight * smooth + detail_weight * detail
    f = lambda v: v.item() if isinstance(v, torch.Tensor) else v
    return total, {"basic_loss": f(basic), "edge_loss": f(edge),
                   "smoothness_loss": f(smooth), "detail_loss": f(detail)}


def thermal_aware_loss_torch(p1, p2, g1, g2, c1=None, c2=None, t1=None, t2=None,
                             alpha=0.2, edge_weight=0.5, smoothness_weight=0.3):
    """v1 loss, utils/loss.py:4-72: edge == smoothness, unpadded diffs, exp(-10|dt|)."""
    basic = confidence_weighted_regression_loss_torch(p1, p2, g1, g2, c1, c2, alpha)
    edge = 0
    if t1 is not None and t2 is not None and isinstance(t1, torch.Tensor) and t1.dim() == 3:
        for p, t in ((p1, t1), (p2, t2)):
            gr, z = _gray_torch(t), p[..., 2]
            tx = (gr[:, 1:] - gr[:, :-1]).abs()
            ty = (gr[1:, :] - gr[:-1, :]).abs()
            ax = (z[:, 1:] - z[:, :-1]).abs()
            ay = (z[1:, :] - z[:-1, :]).abs()
            edge = edge + (ax * torch.exp(-tx * 10)).mean() + (ay * torch.exp(-ty * 10)).mean()
    smooth = edge
    total = basic + edge_weight * edge + smoothness_weight * smooth
    f = lambda v: v.item() if isinstance(v, torch.Tensor) else v
    return total, {"basic_loss": f(basic), "edge_loss": f(edge), "smoothness_loss": f(smooth)}


def batched_loss_torch(P1, P2, G1, G2, C1, C2, T1, T2, **kw):
    """Oracle of OUR batched extension: loop the per-sample reference over the
    batch exactly as train_thermal_dustr.py:182-360 does (skip non-finite or
    <= 0 samples, divide by the number of valid ones).  Returns
    (mean_loss tensor, per-sample [B,5] float64 array: total,basic,edge,smooth,detail, valid[B])."""
    B = P1.shape[0]
    acc, n_valid = 0.0, 0
    rows, valid = [], []
    for b in range(B):
        loss, comp = enhanced_thermal_aware_loss_torch(
            P1[b], P2[b], G1[b], G2[b],
            None if C1 is None else C1[b], None if C2 is None else C2[b],
            None if T1 is None else T1[b], None if T2 is None else T2[b], **kw)
        ok = bool(torch.isfinite(loss) and loss > 0)        # train_thermal_dustr.py:320
        if ok:
            acc = acc + loss
            n_valid += 1
        valid.append(ok)
        rows.append([float(loss.detach()), comp["basic_loss"], comp["edge_loss"],
                     comp["smoothness_loss"], comp["detail_loss"]])
    mean = acc / n_valid if n_valid else torch.zeros(())
    return mean, np.asarray(rows, np.float64), np.asarray(valid)


# --------------------------------------------------------------------------- numpy fp64 closed form
def _gray_np(t):
    t = np.asarray(t)
    if t.shape[0] == 3:
        # keep the reference's fp32 rounding of the gray image (it is an input
        # to everything downstream), then promote
        tf = t.astype(np.float32)
        return (np.float32(GRAY[0]) * tf[0] + np.float32(GRAY[1]) * tf[1]
                + np.float32(GRAY[2]) * tf[2]).astype(np.float64)
    return t[0].astype(np.float64)


def _pool_np(a, s):
    h, w = a.shape[0] // s, a.shape[1] // s
    return a[:h * s, :w * s].reshape(h, s, w, s).mean(axis=(1, 3))


def _pool_f32(a, s):
    """The reference's F.avg_pool2d of an fp32 image, promoted to float64."""
    t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
    return F.avg_pool2d(t[None, None], s, s)[0, 0].numpy().astype(np.float64)


def _sdiff_np(a):
    """signed zero-padded forward differences."""
    dx = np.zeros_like(a)
    dy = np.zeros_like(a)
    dx[:, :-1] = a[:, 1:] - a[:, :-1]
    dy[:-1, :] = a[1:, :] - a[:-1, :]
    return dx, dy


def loss_fwd_bwd_f64(p1, p2, g1, g2, c1=None, c2=None, t1=None, t2=None, alpha=0.2,
                     edge_weight=0.5, smoothness_weight=0.3, detail_weight=0.3,
                     multi_scale=True):
    """float64 forward + closed-form backward (SURVEY.md Appendix A).

    Returns dict(total, basic, edge, smooth, detail, dp1, dp2, dc1, dc2).
    The gray image is rounded to fp32 first (see _gray_np), and the backward of |dz| at scale 2 takes the sign of the
    reference's fp32 pooled differences (see _pool_f32); everything else fp64.
    """
    out = {"basic": 0.0, "edge": 0.0, "smooth": 0.0, "detail": 0.0}
    grads = []
    views = ((p1, g1, c1, t1), (p2, g2, c2, t2))
    have_thermal = t1 is not None and t2 is not None
    for view, (p, g, c, t) in enumerate(views):
        p = np.asarray(p, np.float64)
        g = np.asarray(g, np.float64)
        H, W = p.shape[:2]
        N = H * W
        d = p - g
        l = np.abs(d).sum(-1) / 3.0
        craw = np.ones((H, W)) if c is None else np.asarray(c, np.float64)
        cc = np.clip(craw, np.float32(CONF_MIN).astype(np.float64), CONF_MAX)
        out["basic"] += float((cc * l - alpha * np.log(cc)).mean())
        dp = cc[..., None] * np.sign(d) / (3.0 * N)
        inside = (craw >= np.float32(CONF_MIN).astype(np.float64)) & (craw <= CONF_MAX)
        dc = np.where(inside, (l - alpha / cc) / N, 0.0)
        if have_thermal:
            gr0, z0, gz0 = _gray_np(t), p[..., 2], g[..., 2]
            for s in ([1, 2] if multi_scale else [1]):
                lam = 1.0 if s == 1 else 0.7 / s
                gr, z, gz = (gr0, z0, gz0) if s == 1 else (_pool_np(gr0, s), _pool_np(z0, s), _pool_np(gz0, s))
                h, w_ = z.shape
                n = h * w_
                tx, ty = (np.abs(a) for a in _sdiff_np(gr))
                sx, sy = _sdiff_np(z)
                # d|dz|/dz = sign(dz) of the reference's fp32 pooled image: two cells that pool to the same fp32 value
                # have sign 0 there, whatever their float64 means say (at s == 1 the fp32 signs are already exact)
                gsx, gsy = (sx, sy) if s == 1 else _sdiff_np(_pool_f32(z0, s))
                bx, by = (np.abs(a) for a in _sdiff_np(gz))
                ax, ay = np.abs(sx), np.abs(sy)
                m = CLAMP_VIEW[view]
                wt = np.exp(-THERMAL_FACTOR * np.clip(tx / (tx.mean() + EPS), 0, m)) * \
                    np.exp(-THERMAL_FACTOR * np.clip(ty / (ty.mean() + EPS), 0, m))
                hub = lambda q: np.where(q < HUBER_DELTA, 0.5 * q * q, HUBER_DELTA * (q - 0.5 * HUBER_DELTA))
                out["edge"] += lam * float((ax * (1 - wt)).mean() + (ay * (1 - wt)).mean())
                out["smooth"] += lam * float((ax * ax * wt).mean() + (ay * ay * wt).mean())
                out["detail"] += lam * float(hub(np.abs(ax - bx)).mean() + hub(np.abs(ay - by)).mean())

                def q(sd, a, b):
                    e = a - b
                    dh = np.where(np.abs(e) < HUBER_DELTA, np.abs(e), HUBER_DELTA) * np.sign(e)
                    return (lam / n) * np.sign(sd) * (edge_weight * (1 - wt)
                                                      + smoothness_weight * 2 * a * wt
                                                      + detail_weight * dh)
                qx, qy = q(gsx, ax, bx), q(gsy, ay, by)   # zero on the padded last col / row (sign(0)=0)
                dz = -qx - qy
                dz[:, 1:] += qx[:, :-1]
                dz[1:, :] += qy[:-1, :]
                if s == 1:
                    dp[..., 2] += dz
                else:
                    up = np.repeat(np.repeat(dz, s, 0), s, 1) / (s * s)
                    dp[:h * s, :w_ * s, 2] += up
        grads.append((dp, dc))
    out["total"] = out["basic"] + edge_weight * out["edge"] + smoothness_weight * out["smooth"] \
        + detail_weight * out["detail"]
    out["dp1"], out["dc1"] = grads[0]
    out["dp2"], out["dc2"] = grads[1]
    return out


# --------------------------------------------------------------------------- synthetic inputs (SURVEY.md 8d / Appendix C KAT-L)
def make_kat_inputs(H, W, seed=0):
    """KAT-L generator, SURVEY.md Appendix C (CPU torch.Generator, fixed draw order)."""
    g = torch.Generator().manual_seed(seed)
    gt1 = torch.randn(H, W, 3, generator=g); gt1[..., 2] = gt1[..., 2].abs() * 3 + 1.5
    gt2 = torch.randn(H, W, 3, generator=g); gt2[..., 2] = gt2[..., 2].abs() * 3 + 1.5
    p1 = gt1 + 0.1 * torch.randn(H, W, 3, generator=g)
    p2 = gt2 + 0.1 * torch.randn(H, W, 3, generator=g)
    c1 = 1 + 4 * torch.rand(H, W, generator=g)
    c2 = 1 + 4 * torch.rand(H, W, generator=g)
    t1 = torch.rand(1, H, W, generator=g).repeat(3, 1, 1)
    t2 = torch.rand(1, H, W, generator=g).repeat(3, 1, 1)
    return p1, p2, gt1, gt2, c1, c2, t1, t2


def make_batch_inputs(B, H, W, seed=0, stress_conf=False, smooth=True):
    """Batched synthetic pointmap pairs, SURVEY.md 8(d).  `smooth` thermal gives a
    realistic mix of flat regions and edges (box-blurred noise + steps)."""
    g = torch.Generator().manual_seed(seed)
    G1 = torch.randn(B, H, W, 3, generator=g); G1[..., 2] = 1.5 + 3 * G1[..., 2].abs()
    G2 = torch.randn(B, H, W, 3, generator=g); G2[..., 2] = 1.5 + 3 * G2[..., 2].abs()
    P1 = G1 + 0.1 * torch.randn(B, H, W, 3, generator=g)
    P2 = G2 + 0.1 * torch.randn(B, H, W, 3, generator=g)
    if stress_conf:
        C1 = 12 * torch.rand(B, H, W, generator=g) - 0.5
        C2 = 12 * torch.rand(B, H, W, generator=g) - 0.5
    else:
        C1 = 1 + 4 * torch.rand(B, H, W, generator=g)
        C2 = 1 + 4 * torch.rand(B, H, W, generator=g)
    T = torch.rand(2, B, 1, H, W, generator=g)
    if smooth:
        k = 5
        T = F.avg_pool2d(F.pad(T.reshape(2 * B, 1, H, W), (k // 2,) * 4, mode="replicate"), k, 1)
        T = T.reshape(2, B, 1, H, W)
        T = (T - T.amin()) / (T.amax() - T.amin())
        T[..., : H // 2, : W // 3] = (T[..., : H // 2, : W // 3] * 0.5 + 0.5)
    T1 = T[0].repeat(1, 3, 1, 1).contiguous()
    T2 = T[1].repeat(1, 3, 1, 1).contiguous()
    return P1, P2, G1, G2, C1, C2, T1, T2

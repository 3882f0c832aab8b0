"""Float64 restatement of the reference's ComputeLoss (utils/loss.py:131-244), written out step by step so that it doubles as
the specification of csrc/y3_loss.cu.  Test infrastructure only: nothing under yolov3_b200/ imports it.

Two kinds of arithmetic, kept apart on purpose:
  - every DECISION of build_targets is taken in float32, exactly as the reference takes it: t * gain, the wh ratio and its
    reciprocal, the anchor_t comparison, gxy % 1 < 0.5, gxy > 1, the inverse gxi = n - gxy, the truncating .long() and the
    clamp of the grid indices.  A kernel that matches the reference must take the same branch at every fp32 boundary;
  - every VALUE (CIoU, BCE, the means, the balance and hyp gains) is computed in float64, with autograd for dL/dp, so that
    the float32 reference and the float32 kernel are both compared against something more precise than either.

tobj is written by an explicit loop in the reference's enumeration order (offset-major, then anchor, then target) so that
on a cell several matches share the last one wins, which is what the reference's `tobj[b, a, gj, gi] = iou` does at the
sizes where it is well defined.  tbox is formed from the CLAMPED grid indices: the reference's gi, gj are views of gij and
are clamped in place (loss.py:236-239) one statement before it forms gxy - gij (:240).
"""
from __future__ import annotations

import math

import numpy as np
import torch

OFFSETS = ((0.0, 0.0), (0.5, 0.0), (0.0, 0.5), (-0.5, 0.0), (0.0, -0.5))  # loss.py:192-205, g = 0.5
BALANCE = {3: [4.0, 1.0, 0.4]}  # loss.py:122; any other nl takes the first nl of [4.0, 1.0, 0.25, 0.06, 0.02]


def balance_for(nl):
    return BALANCE.get(nl, [4.0, 1.0, 0.25, 0.06, 0.02])


def build_targets(shapes, targets, anchors, anchor_t=4.0):
    """Matches per level, in the reference's order.  shapes: (bs, na, ny, nx, ...) per level; targets [nt, 6] (img, cls, x,
    y, w, h normalised); anchors [nl, na, 2] in grid units.  Returns one dict per level of int64 arrays b, a, gj, gi, cls
    and float64 arrays tbox [n, 4], anch [n, 2]."""
    t32 = torch.as_tensor(targets, dtype=torch.float32).reshape(-1, 6)
    anchors = torch.as_tensor(anchors, dtype=torch.float32)
    thr = torch.tensor(anchor_t, dtype=torch.float32)
    half = torch.tensor(0.5, dtype=torch.float32)
    one = torch.tensor(1.0, dtype=torch.float32)
    out = []
    for l, shape in enumerate(shapes):
        ny, nx = int(shape[2]), int(shape[3])
        fx, fy = torch.tensor(float(nx)), torch.tensor(float(ny))  # float32 gains
        gx, gy = t32[:, 2] * fx, t32[:, 3] * fy
        gw, gh = t32[:, 4] * fx, t32[:, 5] * fy
        ix, iy = fx - gx, fy - gy
        vals = list(zip(gx.tolist(), gy.tolist(), gw.tolist(), gh.tolist()))  # the float32 values, exactly
        rec = {k: [] for k in ("b", "a", "gj", "gi", "cls", "tbox", "anch")}
        for ox, oy in OFFSETS:
            if ox > 0:
                sel_o = (torch.remainder(gx, one) < half) & (gx > one)
            elif oy > 0:
                sel_o = (torch.remainder(gy, one) < half) & (gy > one)
            elif ox < 0:
                sel_o = (torch.remainder(ix, one) < half) & (ix > one)
            elif oy < 0:
                sel_o = (torch.remainder(iy, one) < half) & (iy > one)
            else:
                sel_o = torch.ones_like(gx, dtype=torch.bool)
            for a in range(anchors.shape[1]):
                aw, ah = anchors[l, a, 0], anchors[l, a, 1]
                rw, rh = gw / aw, gh / ah
                m = torch.maximum(torch.maximum(rw, one / rw), torch.maximum(rh, one / rh))
                gi0 = (gx - torch.tensor(ox)).long().tolist()  # .long() truncates toward zero
                gj0 = (gy - torch.tensor(oy)).long().tolist()
                b, c = t32[:, 0].long().tolist(), t32[:, 1].long().tolist()
                for t in torch.nonzero((m < thr) & sel_o).flatten().tolist():
                    gi, gj = min(max(gi0[t], 0), nx - 1), min(max(gj0[t], 0), ny - 1)
                    rec["b"].append(b[t])
                    rec["cls"].append(c[t])
                    rec["a"].append(a)
                    rec["gi"].append(gi)
                    rec["gj"].append(gj)
                    x, y, w, h = vals[t]
                    rec["tbox"].append((x - gi, y - gj, w, h))
                    rec["anch"].append((float(aw), float(ah)))
        out.append({k: (np.array(v, np.float64).reshape(-1, 4 if k == "tbox" else 2) if k in ("tbox", "anch")
                        else np.array(v, np.int64)) for k, v in rec.items()})
    return out


def ciou(b1, b2, eps=1e-7):
    """bbox_iou(b1, b2, xywh=True, CIoU=True) (ultralytics, called loss.py:151) in the precision of its inputs; alpha is a
    constant of the backward pass as in the original (computed under no_grad)."""
    x1, y1, w1, h1 = b1.unbind(-1)
    x2, y2, w2, h2 = b2.unbind(-1)
    b1x1, b1x2, b1y1, b1y2 = x1 - w1 / 2, x1 + w1 / 2, y1 - h1 / 2, y1 + h1 / 2
    b2x1, b2x2, b2y1, b2y2 = x2 - w2 / 2, x2 + w2 / 2, y2 - h2 / 2, y2 + h2 / 2
    inter = (torch.minimum(b1x2, b2x2) - torch.maximum(b1x1, b2x1)).clamp(0) * (
        torch.minimum(b1y2, b2y2) - torch.maximum(b1y1, b2y1)).clamp(0)
    union = w1 * h1 + w2 * h2 - inter + eps
    iou = inter / union
    cw = torch.maximum(b1x2, b2x2) - torch.minimum(b1x1, b2x1)
    ch = torch.maximum(b1y2, b2y2) - torch.minimum(b1y1, b2y1)
    c2 = cw**2 + ch**2 + eps
    rho2 = ((b2x1 + b2x2 - b1x1 - b1x2) ** 2 + (b2y1 + b2y2 - b1y1 - b1y2) ** 2) / 4
    v = (4 / math.pi**2) * (torch.atan(w2 / h2) - torch.atan(w1 / h1)) ** 2
    with torch.no_grad():
        alpha = v / (v - iou + (1 + eps))
    return iou - (rho2 / c2 + v * alpha)


def bce_logits(x, t, pw):
    """BCEWithLogitsLoss(pos_weight=pw) element-wise: (1 - t) x + (1 + (pw - 1) t) softplus(-x)."""
    lw = 1.0 + (pw - 1.0) * t
    return (1.0 - t) * x + lw * (torch.clamp(-x, min=0) + torch.log1p(torch.exp(-x.abs())))


def compute_loss(p, targets, anchors, hyp, nc=None):
    """ComputeLoss.__call__ (loss.py:131-181; fl_gamma = 0, autobalance off, gr = 1) in float64.  p: raw [bs, na, ny, nx, no]
    per level (any float dtype; gradients are taken w.r.t. a float64 copy).  Returns a dict with loss (float), items
    [3] (lbox, lobj, lcls), grads (float64 dL/dp per level, for an upstream gradient of 1), matches (build_targets per level),
    cells (set of matched (level, b, a, gj, gi)) and tobj (float64 [bs, na, ny, nx] target per level)."""
    nl = len(p)
    nc = p[0].shape[-1] - 5 if nc is None else nc
    ls = hyp.get("label_smoothing", 0.0)
    cp, cn = 1.0 - 0.5 * ls, 0.5 * ls
    balance = balance_for(nl)
    pd = [torch.as_tensor(x).detach().double().requires_grad_(True) for x in p]
    bt = build_targets([tuple(x.shape) for x in pd], targets, anchors, hyp["anchor_t"])
    lbox = lobj = lcls = torch.zeros((), dtype=torch.float64)
    cells, tobjs = set(), []
    for l, pi in enumerate(pd):
        m = bt[l]
        n = len(m["b"])
        tobj = np.zeros(pi.shape[:4], dtype=np.float64)
        if n:
            idx = (torch.from_numpy(m["b"]), torch.from_numpy(m["a"]), torch.from_numpy(m["gj"]), torch.from_numpy(m["gi"]))
            ps = pi[idx]
            pxy = ps[:, 0:2].sigmoid() * 2 - 0.5
            pwh = (ps[:, 2:4].sigmoid() * 2) ** 2 * torch.from_numpy(m["anch"])
            iou = ciou(torch.cat((pxy, pwh), 1), torch.from_numpy(m["tbox"]))
            lbox = lbox + (1.0 - iou).mean()
            iou_t = iou.detach().clamp(0).tolist()
            for k, cell in enumerate(zip(*(v.tolist() for v in idx))):  # reference order; the last write wins
                tobj[cell] = iou_t[k]
                cells.add((l,) + cell)
            if nc > 1:
                tc = torch.full((n, nc), cn, dtype=torch.float64)
                tc[torch.arange(n), torch.from_numpy(m["cls"])] = cp
                lcls = lcls + bce_logits(ps[:, 5:], tc, hyp["cls_pw"]).mean()
        lobj = lobj + bce_logits(pi[..., 4], torch.from_numpy(tobj), hyp["obj_pw"]).mean() * balance[l]
        tobjs.append(tobj)
    lbox, lobj, lcls = lbox * hyp["box"], lobj * hyp["obj"], lcls * hyp["cls"]
    loss = (lbox + lobj + lcls) * pd[0].shape[0]
    loss.backward()
    return dict(loss=float(loss.detach()), items=np.array([float(v.detach()) for v in (lbox, lobj, lcls)]),
                grads=[x.grad.numpy() for x in pd], matches=bt, cells=cells, tobj=tobjs)

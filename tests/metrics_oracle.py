"""CPU restatement of the reference's validation metrics — ap_per_class + compute_ap (utils/metrics.py:22-120) and
ConfusionMatrix.process_batch (utils/metrics.py:134-178) — written out step by step so that it doubles as the specification of
the device kernels in yolov3_b200/csrc/y3_metrics.cu.  Test infrastructure only: nothing under yolov3_b200/ imports it.

What is spelled out rather than delegated to numpy:
  - the order: class, then confidence descending, then input row (a stable sort; numpy's argsort(-conf) at metrics.py:42 is
    unstable, so on bit-equal confidences the reference's order is unspecified);
  - np.interp: j = (number of xp <= x) - 1, i.e. the last duplicate wins; j == -1 -> left, j == len - 1 -> fp[-1],
    xp[j] == x -> fp[j], otherwise slope * (x - xp[j]) + fp[j] with slope = (fp[j+1] - fp[j]) / (xp[j+1] - xp[j]);
  - np.trapezoid over the 101 COCO points: add.reduce(d * (y[1:] + y[:-1]) / 2.0) is numpy's pairwise sum, which for 100 terms
    is eight interleaved partial sums, combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the last four terms in order;
  - smooth(y, 0.1): 101 taps of 1/101 over y padded with 50 copies of each end, summed in tap order (np.convolve goes through
    BLAS ddot, whose order is not specified: the reference may differ from this by a few ulp);
  - ConfusionMatrix ties on bit-equal IoU: the lower label index, then the lower detection index wins.
"""
from __future__ import annotations

import numpy as np
import torch

AP_X = np.array([k * 0.01 for k in range(100)] + [1.0])  # == np.linspace(0, 1, 101)
PX = np.array([k * (1.0 / 999) for k in range(999)] + [1.0])  # == np.linspace(0, 1, 1000)


def interp(x, xp, fp, left=None, right=None):
    """np.interp for nondecreasing xp, restated (x, xp, fp float64 1-D)."""
    x, xp, fp = (np.asarray(v, dtype=np.float64) for v in (x, xp, fp))
    n = xp.shape[0]
    lv = fp[0] if left is None else float(left)
    rv = fp[-1] if right is None else float(right)
    out = np.empty_like(x)
    for i, xv in enumerate(x):
        if xv > xp[-1]:
            out[i] = rv
            continue
        j = int(np.count_nonzero(xp <= xv)) - 1
        if j == -1:
            out[i] = lv
        elif j == n - 1:
            out[i] = fp[j]
        elif xp[j] == xv:
            out[i] = fp[j]
        else:
            slope = (fp[j + 1] - fp[j]) / (xp[j + 1] - xp[j])
            out[i] = slope * (xv - xp[j]) + fp[j]
    return out


def pairwise_sum(a):
    """numpy's pairwise summation of a contiguous float64 array of at most 128 elements."""
    a = np.asarray(a, dtype=np.float64)
    n = a.shape[0]
    assert n <= 128
    if n < 8:
        res = 0.0
        for v in a:
            res += v
        return res
    r = [a[q] for q in range(8)]
    i = 8
    while i < n - n % 8:
        for q in range(8):
            r[q] += a[i + q]
        i += 8
    res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    for k in range(i, n):
        res += a[k]
    return res


def trapezoid(y, x):
    """np.trapezoid(y, x) for 1-D inputs of at most 129 points."""
    y, x = np.asarray(y, dtype=np.float64), np.asarray(x, dtype=np.float64)
    terms = [(x[i + 1] - x[i]) * (y[i + 1] + y[i]) / 2.0 for i in range(len(y) - 1)]
    return pairwise_sum(np.array(terms))


def compute_ap(recall, precision):
    """compute_ap (metrics.py:94-120), method 'interp'."""
    mrec = np.concatenate(([0.0], recall, [1.0]))
    mpre = np.concatenate(([1.0], precision, [0.0]))
    env = mpre.copy()
    for i in range(len(env) - 2, -1, -1):  # suffix maximum: the precision envelope
        env[i] = max(env[i], env[i + 1])
    return trapezoid(interp(AP_X, mrec, env), AP_X)


def smooth(y, f=0.1):
    nf = round(len(y) * f * 2) // 2 + 1
    yp = np.concatenate((np.full(nf // 2, y[0]), y, np.full(nf // 2, y[-1])))
    w = 1.0 / nf
    acc = np.zeros(len(y))
    for t in range(nf):
        acc = acc + yp[t:t + len(y)] * w
    return acc


def ap_per_class(tp, conf, pred_cls, target_cls, eps=1e-16, nc=None):
    """ap_per_class (metrics.py:22-91) by class id.  Returns a dict of arrays indexed by class id 0..nc-1 (ap [nc, niou]; p, r,
    f1, tp, fp at the chosen F1 index; nt; present) plus the index itself (`i`), the smoothed mean-F1 curve (`f1_smooth`) and
    the reference's own tuple (`ref`: tp, fp, p, r, f1, ap, classes over the present classes only)."""
    tp = np.asarray(tp).astype(bool).reshape(len(conf), -1)
    conf = np.asarray(conf, dtype=np.float32)
    pred_cls = np.asarray(pred_cls, dtype=np.float32)
    target_cls = np.asarray(target_cls, dtype=np.float32)
    niou = tp.shape[1]
    if nc is None:
        nc = int(target_cls.max()) + 1 if len(target_cls) else 1
    order = np.argsort(-conf, kind="stable")  # conf descending, ties by row
    tp, conf, pred_cls = tp[order], conf[order], pred_cls[order]
    nt = np.array([int(np.count_nonzero(target_cls == c)) for c in range(nc)], dtype=np.int64)
    present = nt > 0
    ap = np.zeros((nc, niou))
    pc, rc = np.zeros((nc, 1000)), np.zeros((nc, 1000))
    for c in range(nc):
        sel = pred_cls == c
        n_l, n_p = int(nt[c]), int(np.count_nonzero(sel))
        if n_l == 0 or n_p == 0:
            continue
        t = tp[sel].astype(np.int64)
        tpc = np.cumsum(t, 0)
        fpc = np.cumsum(1 - t, 0)
        recall = tpc / (n_l + eps)
        precision = tpc / (tpc + fpc)
        xp = -conf[sel].astype(np.float64)
        rc[c] = interp(-PX, xp, recall[:, 0], left=0)
        pc[c] = interp(-PX, xp, precision[:, 0], left=1)
        for j in range(niou):
            ap[c, j] = compute_ap(recall[:, j], precision[:, j])
    f1c = 2 * pc * rc / (pc + rc + eps)
    mean = np.zeros(1000)
    for c in np.flatnonzero(present):  # f1.mean(0): rows added in class order
        mean = mean + f1c[c]
    with np.errstate(invalid="ignore"):
        mean = mean / int(present.sum())
    fs = smooth(mean, 0.1)
    i = int(np.argmax(fs))
    p, r, f1 = pc[:, i] * present, rc[:, i] * present, f1c[:, i] * present
    tpo = np.round(r * nt)
    fpo = np.round(tpo / (p + eps) - tpo)
    cls = np.flatnonzero(present)
    return {"ap": ap, "p": p, "r": r, "f1": f1, "tp": tpo, "fp": fpo, "nt": nt, "present": present, "i": i, "f1_smooth": fs,
            "pcurve": pc, "rcurve": rc,
            "ref": (tpo[cls], fpo[cls], p[cls], r[cls], f1[cls], ap[cls], cls.astype(int))}


def box_iou(box1, box2, eps=1e-7):
    """box_iou in fp32, the reference's operand order: inter / (a1 + a2 - inter + eps), [N, M]."""
    b1, b2 = torch.as_tensor(box1).float(), torch.as_tensor(box2).float()
    lt = torch.max(b1[:, None, :2], b2[None, :, :2])
    rb = torch.min(b1[:, None, 2:], b2[None, :, 2:])
    inter = (rb - lt).clamp(min=0).prod(2)
    a1 = (b1[:, 2] - b1[:, 0]) * (b1[:, 3] - b1[:, 1])
    a2 = (b2[:, 2] - b2[:, 0]) * (b2[:, 3] - b2[:, 1])
    return (inter / (a1[:, None] + a2[None, :] - inter + eps)).numpy()


def _cls(v, nc):
    c = int(v)  # tensor.int(): truncation
    return c if 0 <= c < nc and v > -1 else None


def confusion_update(matrix, detections, labels, nc, conf=0.25, iou_thres=0.45):
    """ConfusionMatrix.process_batch (metrics.py:134-178) on one image, accumulating into matrix [nc+1, nc+1] (int64).
    detections [N, 6] (xyxy, conf, cls) or None; labels [M, 5] (cls, xyxy), or the class vector when detections is None.
    Returns the number of class ids outside [0, nc) that were skipped."""
    invalid = 0
    labels = np.asarray(labels, dtype=np.float32)
    if detections is None:
        for v in labels.reshape(-1, labels.shape[-1] if labels.ndim > 1 else 1)[:, 0]:
            g = _cls(v, nc)
            if g is None:
                invalid += 1
            else:
                matrix[nc, g] += 1
        return invalid
    det = np.asarray(detections, dtype=np.float32)
    det = det[det[:, 4] > np.float32(conf)]
    iou = box_iou(labels[:, 1:], det[:, :4])  # [M, N]
    thr = np.float32(iou_thres)
    # each detection: its highest-IoU label with IoU > thr (np.argmax: the lower label index on ties)
    cand = np.where(iou > thr, iou, -np.inf)
    best_l = np.where(np.isfinite(cand).any(0), np.argmax(cand, 0), -1) if len(labels) else np.full(len(det), -1)
    # each label: the highest-IoU detection among those whose best label it is (the lower detection index on ties)
    best_d = np.full(len(labels), -1)
    for l in range(len(labels)):
        mine = np.flatnonzero(best_l == l)
        if len(mine):
            best_d[l] = mine[np.argmax(iou[l, mine])]
    any_match = bool((best_l >= 0).any())
    for l in range(len(labels)):
        g = _cls(labels[l, 0], nc)
        row = _cls(det[best_d[l], 5], nc) if best_d[l] >= 0 else nc
        if g is None or row is None:
            invalid += 1
        else:
            matrix[row, g] += 1
    if any_match:  # metrics.py:175: unmatched detections count only when the image has a match
        matched = set(int(d) for d in best_d if d >= 0)
        for d in range(len(det)):
            if d in matched:
                continue
            dc = _cls(det[d, 5], nc)
            if dc is None:
                invalid += 1
            else:
                matrix[dc, nc] += 1
    return invalid


def synth_stats(n, nc, n_targets, niou=10, seed=0, p_tp=0.35, classes=None, ties=False):
    """Seeded (tp, conf, pred_cls, target_cls) for ap_per_class: per class at most n_l true positives at threshold 0 and
    fewer at each stricter threshold (what process_batch produces); true positives lean to high confidence.  Confidences are
    distinct float32 values unless `ties`."""
    rng = np.random.default_rng(seed)
    classes = np.arange(nc) if classes is None else np.asarray(classes)
    target_cls = rng.choice(classes, n_targets).astype(np.float32)
    pred_cls = rng.choice(classes, n).astype(np.float32)
    if ties:
        conf = (rng.integers(1, 40, n) / 40.0).astype(np.float32)
    else:
        conf = ((rng.permutation(n) + 0.5) / n).astype(np.float32)
    tp = np.zeros((n, niou), dtype=bool)
    cand = rng.random(n) < p_tp * (0.4 + conf)
    for c in classes:
        rows = np.flatnonzero((pred_cls == c) & cand)
        cap = int(np.count_nonzero(target_cls == c))
        if len(rows) > cap:
            rows = rng.choice(rows, cap, replace=False)
        tp[rows, 0] = True
    for j in range(1, niou):
        tp[:, j] = tp[:, j - 1] & (rng.random(n) < 0.88)
    return tp, conf, pred_cls, target_cls

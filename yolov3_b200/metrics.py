"""Validation metrics on the device — the reference's ``ap_per_class`` (utils/metrics.py:22, with ``compute_ap`` :94) and
``ConfusionMatrix`` (utils/metrics.py:124), called by val.py:340,390,406,424-426.

``ap_per_class`` is the drop-in: the reference's arguments and return tuple (numpy, same dtypes and shapes), computed by
``y3_ap_per_class`` (csrc/y3_metrics.cu) after the inputs are moved to the current CUDA device; one device->host copy of the
small per-class results.  ``ap_per_class_batched`` is the sync-free form: it reads the padded outputs of ``nms_batched`` and
``process_batch_batched`` (concatenated over batches) in place and returns device tensors indexed by class id.
``ConfusionMatrix`` accumulates on the device (``y3_confusion_update``); ``matrix`` copies it to the host.

Parity: AP is bit-identical to the reference; P / R / F1 agree to ~1e-16 (the reference's ``smooth`` sums through BLAS ddot,
whose order is unspecified).  On bit-equal confidences the reference's order is unspecified (an unstable argsort); here rows
of equal confidence keep their input order.  ConfusionMatrix ties on bit-equal IoU: the lower label index, then the lower
detection index wins.  Class ids outside ``[0, nc)`` are counted (``status`` / ``invalid``), never used as an index.
"""
from __future__ import annotations

import logging
import warnings
from typing import NamedTuple

import numpy as np
import torch

from . import _lib
from .tensors import _stream

LOGGER = logging.getLogger("yolov3_b200")
MAX_LABELS_PER_IMAGE = 1024  # ConfusionMatrix: labels of one image matched (the rest are reported, see ConfusionMatrix.invalid)


class APResult(NamedTuple):
    """Device tensors indexed by class id 0..nc-1 (rows of classes that are not ``present`` are zero)."""

    tp: torch.Tensor        # float64 [nc] true positives at the F1 index
    fp: torch.Tensor        # float64 [nc] false positives at the F1 index
    p: torch.Tensor         # float64 [nc]
    r: torch.Tensor         # float64 [nc]
    f1: torch.Tensor        # float64 [nc]
    ap: torch.Tensor        # float64 [nc, niou]
    nt: torch.Tensor        # int64 [nc] labels per class
    present: torch.Tensor   # bool [nc]: the class occurs in the targets (the reference's unique_classes)
    f1_index: torch.Tensor  # int32 [1]: index into np.linspace(0, 1, 1000) of the smoothed mean-F1 maximum
    status: torch.Tensor    # int32 [3]: prediction rows / target labels with a class outside [0, nc), curves with tp > labels


def _ap(conf, conf_stride, cls, cls_stride, tp, niou, n, counts, rows_per_image, tcls, tcls_stride, n_targets, nc, eps,
        device) -> APResult:
    L = _lib.lib()
    ws_bytes = L.y3_ap_per_class_workspace_bytes(n, n_targets, niou, nc)
    if ws_bytes < 0:
        raise ValueError(f"ap_per_class: bad sizes (n={n}, n_targets={n_targets}, niou={niou}, nc={nc})")
    ws = torch.empty(max(int(ws_bytes), 1), dtype=torch.uint8, device=device)
    f64 = dict(dtype=torch.float64, device=device)
    out = APResult(torch.empty(nc, **f64), torch.empty(nc, **f64), torch.empty(nc, **f64), torch.empty(nc, **f64),
                   torch.empty(nc, **f64), torch.empty(nc, niou, **f64), torch.empty(nc, dtype=torch.int64, device=device),
                   torch.empty(nc, dtype=torch.bool, device=device), torch.empty(1, dtype=torch.int32, device=device),
                   torch.empty(3, dtype=torch.int32, device=device))
    _lib.check(L.y3_ap_per_class(conf, conf_stride, cls, cls_stride, tp, niou, n, counts, rows_per_image, tcls, tcls_stride,
                                 n_targets, nc, float(eps), ws.data_ptr(), ws.numel(), out.ap.data_ptr(), out.p.data_ptr(),
                                 out.r.data_ptr(), out.f1.data_ptr(), out.tp.data_ptr(), out.fp.data_ptr(), out.nt.data_ptr(),
                                 out.present.data_ptr(), out.f1_index.data_ptr(), out.status.data_ptr(), _stream()),
               "y3_ap_per_class")
    return out


def ap_per_class_batched(det: torch.Tensor, counts: torch.Tensor | None, correct: torch.Tensor, labels: torch.Tensor, nc: int,
                         eps: float = 1e-16) -> APResult:
    """ap_per_class over a padded layout without any host synchronisation.

    det: [N, max_det, 6] (xyxy, conf, cls) — ``nms_batched`` outputs concatenated over batches (only conf and cls are read);
    counts: [N] valid rows per image (None: every row is valid); correct: [N, max_det, niou] bool (``process_batch_batched``);
    labels: collated [nl, 6] = (image, cls, xyxy), or any [nl, k >= 2] whose column 1 is the class; nc: number of classes."""
    assert det.is_cuda and det.dtype == torch.float32 and det.dim() == 3 and det.shape[2] == 6 and det.is_contiguous(), \
        "det: contiguous CUDA fp32 [N, max_det, 6] (yolov3_b200 has no CPU path)"
    nimg, max_det, _ = det.shape
    assert correct.is_cuda and correct.dim() == 3 and correct.shape[:2] == det.shape[:2], "correct: [N, max_det, niou]"
    tp = correct.contiguous().view(torch.uint8) if correct.dtype == torch.bool else correct.to(torch.uint8).contiguous()
    labels = labels.to(det.device, torch.float32).contiguous()
    if labels.dim() == 1:
        labels = labels.reshape(-1, 6)
    if counts is not None:
        counts = counts.to(det.device, torch.int32).contiguous()
        assert counts.numel() == nimg, "counts: one per image"
    n = nimg * max_det
    return _ap(det.data_ptr() + 16, 6, det.data_ptr() + 20, 6, tp.data_ptr() if n else None, tp.shape[2], n,
               counts.data_ptr() if counts is not None else None, max(max_det, 1),
               labels.data_ptr() + 4 if labels.shape[0] else None, labels.shape[1], labels.shape[0], int(nc), eps, det.device)


def ap_per_class(tp, conf, pred_cls, target_cls, plot=False, save_dir=".", names=(), eps=1e-16, prefix=""):
    """Drop-in for utils/metrics.py:22.  tp [n, niou] bool, conf [n], pred_cls [n], target_cls [nt] — numpy arrays (copied to
    the current CUDA device) or CUDA tensors.  Returns (tp, fp, p, r, f1, ap, unique_classes) as the reference does.
    Confidences are evaluated in float32 (what val.py collects); target classes must be integral and >= 0."""
    if plot:
        raise NotImplementedError("ap_per_class(plot=True): plotting is not part of yolov3_b200")
    del save_dir, names, prefix  # used by the reference's plots only
    dev = torch.device("cuda", torch.cuda.current_device())

    def dev_tensor(x, dtype):
        t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
        assert t.device.type in ("cuda", "cpu"), t.device
        return t.to(dev if t.device.type == "cpu" else t.device, dtype).contiguous()

    tpt = dev_tensor(tp, torch.uint8)
    n = tpt.shape[0]
    if tpt.dim() == 1:  # a single IoU threshold given as [n]
        tpt = tpt.reshape(n, 1)
    conf_t, cls_t = dev_tensor(conf, torch.float32).reshape(-1), dev_tensor(pred_cls, torch.float32).reshape(-1)
    tcls = dev_tensor(target_cls, torch.float32).reshape(-1)
    assert conf_t.numel() == n and cls_t.numel() == n, "tp, conf and pred_cls must have one row per detection"
    if tcls.numel():
        lo, hi = torch.stack(torch.aminmax(tcls)).tolist()  # one small copy: the class count sizes the outputs
        if not (lo >= 0 and np.isfinite(hi)):
            raise ValueError(f"ap_per_class: target classes must be finite and >= 0 (got [{lo}, {hi}])")
        nc = int(hi) + 1
    else:
        nc = 1
    res = _ap(conf_t.data_ptr() if n else None, 1, cls_t.data_ptr() if n else None, 1, tpt.data_ptr() if n else None,
              max(tpt.shape[1], 1), n, None, max(n, 1), tcls.data_ptr() if tcls.numel() else None, 1, tcls.numel(), nc, eps,
              tpt.device)
    h = {k: v.cpu().numpy() for k, v in res._asdict().items()}
    if h["status"][1]:
        raise ValueError(f"ap_per_class: {h['status'][1]} target classes are not integral class ids")
    if h["status"][2]:
        warnings.warn(f"ap_per_class: {h['status'][2]} (class, threshold) curves have more true positives than labels; "
                      "their AP is not defined by the reference (a non-monotone recall curve)")
    cls = np.flatnonzero(h["present"])
    return h["tp"][cls], h["fp"][cls], h["p"][cls], h["r"][cls], h["f1"][cls], h["ap"][cls], cls.astype(int)


class ConfusionMatrix:
    """Drop-in for utils/metrics.py:124, accumulated on the device: ``matrix`` is [nc+1, nc+1] float64, indexed [pred, true],
    with the background row / column last."""

    def __init__(self, nc, conf=0.25, iou_thres=0.45):
        self.nc = int(nc)
        self.conf = conf
        self.iou_thres = iou_thres
        self._m = None       # int64 [(nc+1)^2] on the device, allocated on first use
        self._status = None  # int32 [2]: class ids outside [0, nc), labels beyond MAX_LABELS_PER_IMAGE in one image

    def _buffers(self, device):
        if self._m is None:
            self._m = torch.zeros((self.nc + 1) ** 2, dtype=torch.int64, device=device)
            self._status = torch.zeros(2, dtype=torch.int32, device=device)
        return self._m, self._status

    def process_batch_batched(self, det: torch.Tensor, counts: torch.Tensor | None, labels: torch.Tensor):
        """A padded batch: det [bs, max_det, 6] (xyxy, conf, cls) + counts [bs] (``nms_batched``), labels [nl, 6] =
        (image, cls, xyxy) in det's coordinate space.  Same as process_batch per image with labels, in image order (an image
        without detections counts its labels as background; one without labels adds nothing).  No host synchronisation."""
        assert det.is_cuda and det.dtype == torch.float32 and det.dim() == 3 and det.shape[2] == 6 and det.is_contiguous(), \
            "det: contiguous CUDA fp32 [bs, max_det, 6] (yolov3_b200 has no CPU path)"
        bs, max_det, _ = det.shape
        labels = labels.to(det.device, torch.float32).contiguous().reshape(-1, 6)
        if counts is not None:
            counts = counts.to(det.device, torch.int32).contiguous()
        m, st = self._buffers(det.device)
        _lib.check(_lib.lib().y3_confusion_update(det.data_ptr(), counts.data_ptr() if counts is not None else None, bs, max_det,
                                                  max_det, labels.data_ptr() if labels.shape[0] else None, labels.shape[0],
                                                  self.nc, float(self.conf), float(self.iou_thres), 1e-7, m.data_ptr(),
                                                  st.data_ptr(), _stream()), "y3_confusion_update")

    def process_batch(self, detections, labels):
        """One image (val.py:390,406): detections [N, 6] (xyxy, conf, cls) and labels [M, 5] (cls, xyxy); or
        detections=None and labels = the class vector [M] (every label a background false negative)."""
        if detections is None:
            cls = torch.as_tensor(labels).reshape(-1)
            dev = cls.device if cls.is_cuda else torch.device("cuda", torch.cuda.current_device())
            lab = torch.zeros(cls.numel(), 6, dtype=torch.float32, device=dev)
            lab[:, 1] = cls.to(dev, torch.float32)
            det = torch.zeros(1, 0, 6, dtype=torch.float32, device=dev)
            return self.process_batch_batched(det, None, lab)
        assert detections.is_cuda, "yolov3_b200 has no CPU path: detections must be a CUDA tensor"
        n = detections.shape[0]
        det = detections.detach().float().contiguous().view(1, n, 6)
        lab = torch.cat((torch.zeros(labels.shape[0], 1, device=det.device), labels.to(det.device).float()), 1)
        return self.process_batch_batched(det, None, lab)

    @property
    def matrix(self) -> np.ndarray:
        if self._m is None:
            return np.zeros((self.nc + 1, self.nc + 1))
        return self._m.cpu().numpy().reshape(self.nc + 1, self.nc + 1).astype(np.float64)

    @property
    def invalid(self) -> tuple[int, int]:
        """(class ids outside [0, nc) that were skipped, labels beyond MAX_LABELS_PER_IMAGE in one image that were ignored)."""
        if self._status is None:
            return 0, 0
        a, b = self._status.tolist()
        return a, b

    def tp_fp(self):
        m = self.matrix
        tp = m.diagonal()
        fp = m.sum(1) - tp
        return tp[:-1], fp[:-1]  # background class removed

    def plot(self, normalize=True, save_dir="", names=()):
        raise NotImplementedError("ConfusionMatrix.plot: plotting is not part of yolov3_b200")

    def print(self):
        m = self.matrix
        for i in range(self.nc + 1):
            LOGGER.info(" ".join(map(str, m[i])))

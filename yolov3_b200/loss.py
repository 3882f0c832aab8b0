"""``ComputeLoss`` and ``box_iou`` — same call contract as the reference (utils/loss.py:98-181, utils/metrics.py:10),
computed by csrc/y3_loss.cu / y3_iou.cu.  The loss kernel produces dL/dp together with the loss, so ``loss.backward()``
costs nothing more than handing those gradients to autograd."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .tensors import _stream


def smooth_bce(eps=0.1):
    """ultralytics smooth_bce (utils/loss.py:114): positive / negative BCE targets under label smoothing."""
    return 1.0 - 0.5 * eps, 0.5 * eps


def box_iou(box1: torch.Tensor, box2: torch.Tensor, eps: float = 1e-7) -> torch.Tensor:
    """IoU of every box1[N,4] with every box2[M,4] (xyxy) -> [N,M] (reference utils/metrics.py:10, val.py:176)."""
    assert box1.is_cuda and box2.is_cuda, "yolov3_b200 has no CPU path"
    b1, b2 = box1.detach().float().contiguous(), box2.detach().float().contiguous()
    out = torch.empty(b1.shape[0], b2.shape[0], dtype=torch.float32, device=b1.device)
    _lib.check(_lib.lib().y3_box_iou(b1.data_ptr(), b1.shape[0], b2.data_ptr(), b2.shape[0], float(eps), out.data_ptr(),
                                     _stream()), "y3_box_iou")
    return out


class _LossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, owner, targets, *p):
        out, grads = owner._run(p, targets, want_grad=any(x.requires_grad for x in p))
        ctx.grads = grads
        ctx.n = len(p)
        return out[0:1].clone(), out[1:4].clone()

    @staticmethod
    def backward(ctx, g_loss, g_items):
        if ctx.grads is None:
            return (None, None) + (None,) * ctx.n
        return (None, None) + tuple(g * g_loss for g in ctx.grads)


class ComputeLoss:
    """Drop-in for utils/loss.py:98.  ``model`` needs ``.hyp`` and a Detect info at ``.model[-1]`` (na, nc, nl, anchors)."""

    sort_obj_iou = False

    def __init__(self, model, autobalance=False):
        if autobalance:
            raise NotImplementedError("autobalance is off in every shipped configuration and is not accelerated")
        h = model.hyp
        if h.get("fl_gamma", 0.0) > 0:
            raise NotImplementedError("focal loss (fl_gamma > 0) is not part of the accelerated path (SURVEY §2.1)")
        m = model.model[-1]
        self.hyp = h
        self.cp, self.cn = smooth_bce(eps=h.get("label_smoothing", 0.0))
        self.balance = {3: [4.0, 1.0, 0.4]}.get(m.nl, [4.0, 1.0, 0.25, 0.06, 0.02])  # utils/loss.py:122
        self.gr, self.autobalance = 1.0, False
        self.na, self.nc, self.nl = m.na, m.nc, m.nl
        if not (1 <= self.nl <= _lib.MAX_LEVELS and 1 <= self.na <= _lib.MAX_ANCHORS):
            raise ValueError(f"loss: nl={self.nl}, na={self.na}; the kernel takes 1..{_lib.MAX_LEVELS} levels of "
                             f"1..{_lib.MAX_ANCHORS} anchors")
        self.anchors = m.anchors.detach().float().cpu()
        self._ws = None

    def _run(self, p, targets, want_grad=True):
        dev = p[0].device
        assert dev.type == "cuda", "yolov3_b200 has no CPU path"
        p = [x.detach().float().contiguous() for x in p]
        t = targets.detach().to(dev).float().contiguous()
        d = _lib.LossDesc()
        d.nl, d.bs, d.na, d.nc = self.nl, p[0].shape[0], self.na, self.nc
        grads = [torch.empty_like(x) for x in p] if want_grad else None
        for l, x in enumerate(p):
            assert x.shape[1] == self.na and x.shape[4] == self.nc + 5
            d.p[l] = x.data_ptr()
            d.grad[l] = grads[l].data_ptr() if want_grad else None
            d.ny[l], d.nx[l] = x.shape[2], x.shape[3]
            d.balance[l] = self.balance[l]
            for a in range(self.na):
                d.anchors[l][a][0], d.anchors[l][a][1] = float(self.anchors[l, a, 0]), float(self.anchors[l, a, 1])
        d.targets, d.nt = (t.data_ptr() if t.shape[0] else None), t.shape[0]
        h = self.hyp
        d.box, d.obj, d.cls = h["box"], h["obj"], h["cls"]
        d.cls_pw, d.obj_pw, d.anchor_t = h["cls_pw"], h["obj_pw"], h["anchor_t"]
        d.cp, d.cn, d.grad_scale = self.cp, self.cn, 1.0
        L = _lib.lib()
        need = L.y3_loss_workspace_bytes(C.byref(d))
        if self._ws is None or self._ws.numel() < need or self._ws.device != dev:
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        out = torch.empty(4, dtype=torch.float32, device=dev)
        _lib.check(L.y3_loss_fwd_bwd(C.byref(d), self._ws.data_ptr(), self._ws.numel(), out.data_ptr(), _stream()),
                   "y3_loss_fwd_bwd")
        self._keep = (p, t)
        return out, grads

    def __call__(self, p, targets):
        """Returns (loss[1] (differentiable w.r.t. p), loss_items[3] = (lbox, lobj, lcls) detached) — loss.py:181."""
        loss, items = _LossFn.apply(self, targets, *p)
        return loss, items.detach()

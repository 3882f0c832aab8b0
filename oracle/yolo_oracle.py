"""TEST INFRASTRUCTURE ONLY — CPU oracle for the YOLOv3 detection hot path.

A plain torch-CPU/numpy *restatement* of the reference algorithm for the path BASELINE.json names
(Model.forward -> Detect decode -> non_max_suppression; ComputeLoss/build_targets), written from the reference's
behaviour, each function citing the reference file:line it follows.  It is the checker for the CUDA path:
only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` leg may import it.
The product package ``yolov3_b200`` never imports anything from ``oracle/``.

Pinning: the reference ships no tests/golden vectors (SURVEY.md §4).  This oracle is pinned against the reference
ITSELF, imported in the build container through ``oracle/ref_shim.py``: ``tests/golden/make_golden.py`` runs
reference and oracle on the same seeded inputs, asserts agreement and writes the fixtures in ``tests/golden/``;
``tests/test_oracle_golden.py`` re-checks the oracle against those committed fixtures on every run.

Third-party arithmetic that is NOT in /root/reference (named + version floor, restated from published formulas):
  * ultralytics>=8.4.110 (requirements.txt:18): bbox_iou(CIoU), box_iou, smooth_bce, xywh2xyxy, fuse_conv_and_bn,
    initialize_weights (BN eps=1e-3, momentum=0.03), make_divisible.
  * torchvision>=0.9 ``ops.nms`` (utils/general.py:733): greedy NMS, strict ``>`` IoU test, stable score sort.
"""
from __future__ import annotations

import math
from pathlib import Path

import numpy as np
import torch
import torch.nn.functional as F
import yaml

BN_EPS = 1e-3  # ultralytics initialize_weights, called models/yolo.py:229


# ----------------------------------------------------------------------------------------------------------------------
# Graph: YAML -> flat node list (restates parse_model, models/yolo.py:298-380, for the module types the shipped
# YAMLs use: Conv, Bottleneck, SPP, nn.MaxPool2d, nn.ZeroPad2d, nn.Upsample, Concat, Detect)
# ----------------------------------------------------------------------------------------------------------------------
def make_divisible(x, d):
    return math.ceil(x / d) * d


def load_cfg(cfg):
    if isinstance(cfg, dict):
        return cfg
    with open(cfg, encoding="ascii", errors="ignore") as f:
        return yaml.safe_load(f)


def parse_graph(cfg, ch=3):
    """Return (nodes, save).  Each node: dict(i, f, type, n, args, c_in, c_out).  models/yolo.py:298-380."""
    d = load_cfg(cfg)
    anchors, nc, gd, gw = d["anchors"], d["nc"], d["depth_multiple"], d["width_multiple"]
    na = len(anchors[0]) // 2
    no = na * (nc + 5)
    chs, nodes, save = [ch], [], []
    c2 = ch
    for i, (f, n, m, args) in enumerate(d["backbone"] + d["head"]):
        m = m.replace("nn.", "")
        args = [nc if a == "nc" else anchors if a == "anchors" else (None if a == "None" else a) for a in args]
        n = max(round(n * gd), 1) if n > 1 else n
        if m in ("Conv", "Bottleneck", "SPP"):
            c1, c2 = chs[f], args[0]
            if c2 != no:
                c2 = make_divisible(c2 * gw, 8)
            args = [c1, c2, *args[1:]]
        elif m == "Concat":
            c1 = [chs[x] for x in f]
            c2 = sum(c1)
        elif m == "Detect":
            c1 = [chs[x] for x in f]
            args = [nc, anchors, c1]
        elif m in ("MaxPool2d", "ZeroPad2d", "Upsample"):
            c1 = c2 = chs[f]
        else:
            raise NotImplementedError(f"module {m} is not used by the shipped yolov3 YAMLs")
        nodes.append(dict(i=i, f=f, type=m, n=n, args=args, c_in=c1, c_out=c2))
        save.extend(x % i for x in ([f] if isinstance(f, int) else f) if x != -1)
        if i == 0:
            chs = []
        chs.append(c2)
    return nodes, sorted(save)


# ----------------------------------------------------------------------------------------------------------------------
# Parameters: same names as the reference state_dict (model.<i>[.<j>].cv1.conv.weight ...)
# ----------------------------------------------------------------------------------------------------------------------
def _conv_names(prefix):
    return prefix + ".conv.weight", prefix + ".bn"


def conv_prefixes(nodes):
    """List (prefix, c1, c2, k, s) for every Conv+BN block in reference module order, and detect heads."""
    out = []
    for nd in nodes:
        base = f"model.{nd['i']}"
        reps = [base] if nd["n"] == 1 else [f"{base}.{j}" for j in range(nd["n"])]
        if nd["type"] == "Conv":
            c1, c2, *rest = nd["args"]
            k = rest[0] if len(rest) > 0 else 1
            s = rest[1] if len(rest) > 1 else 1
            for r in reps:
                out.append((r, c1, c2, k, s))
        elif nd["type"] == "Bottleneck":
            c1, c2, *rest = nd["args"]
            c_ = int(c2 * 0.5)
            for r in reps:
                out.append((r + ".cv1", c1, c_, 1, 1))
                out.append((r + ".cv2", c_, c2, 3, 1))
                c1 = c2
        elif nd["type"] == "SPP":
            c1, c2, *rest = nd["args"]
            ks = rest[0] if rest else (5, 9, 13)
            c_ = c1 // 2
            out.append((base + ".cv1", c1, c_, 1, 1))
            out.append((base + ".cv2", c_ * (len(ks) + 1), c2, 1, 1))
    return out


def detect_strides(nodes, ch=3):
    """Strides the reference probes with a 256x256 forward (models/yolo.py:222); derived here from the graph."""
    scale = []  # down-sampling factor of every node's output relative to the network input
    for nd in nodes:
        i, f = nd["i"], nd["f"]

        def src(j):
            return 1.0 if i == 0 else scale[j if j >= 0 else i + j]

        if nd["type"] == "Detect":
            return [scale[x] for x in f]
        s = src(f[0]) if nd["type"] == "Concat" else src(f)
        if nd["type"] == "Conv":
            s *= nd["args"][3] if len(nd["args"]) > 3 else 1
        elif nd["type"] == "MaxPool2d":
            s *= nd["args"][1] if len(nd["args"]) > 1 else nd["args"][0]
        elif nd["type"] == "Upsample":
            s /= nd["args"][1]
        scale.append(s)
    raise ValueError("graph has no Detect node")


def init_params(cfg, seed=0, randomize_bn=True, ch=3):
    """Random-init parameters with the reference's init statistics (models/yolo.py:193-231,282-292).

    Conv2d: PyTorch default kaiming-uniform(a=sqrt(5)) == U(-1/sqrt(fan_in), 1/sqrt(fan_in)); BN: gamma=1, beta=0,
    mean=0, var=1 unless ``randomize_bn`` (SURVEY §8(d) config 2: mean~N(0,.1) var~U(.5,1.5) gamma~U(.5,1.5)
    beta~N(0,.1) so that the BN fold is non-trivial).  Detect bias: obj += log(8/(640/s)^2), cls += log(0.6/(nc-0.99999)).
    """
    d = load_cfg(cfg)
    nodes, _ = parse_graph(d, ch)
    g = torch.Generator().manual_seed(seed)
    p = {}
    for prefix, c1, c2, k, s in conv_prefixes(nodes):
        bound = 1.0 / math.sqrt(c1 * k * k)
        p[prefix + ".conv.weight"] = (torch.rand(c2, c1, k, k, generator=g) * 2 - 1) * bound
        if randomize_bn:
            p[prefix + ".bn.weight"] = torch.rand(c2, generator=g) + 0.5
            p[prefix + ".bn.bias"] = torch.randn(c2, generator=g) * 0.1
            p[prefix + ".bn.running_mean"] = torch.randn(c2, generator=g) * 0.1
            p[prefix + ".bn.running_var"] = torch.rand(c2, generator=g) + 0.5
        else:
            p[prefix + ".bn.weight"] = torch.ones(c2)
            p[prefix + ".bn.bias"] = torch.zeros(c2)
            p[prefix + ".bn.running_mean"] = torch.zeros(c2)
            p[prefix + ".bn.running_var"] = torch.ones(c2)
    det = nodes[-1]
    nc, anchors, chs = det["args"]
    na = len(anchors[0]) // 2
    no = nc + 5
    strides = detect_strides(nodes, ch)
    a = torch.tensor(anchors, dtype=torch.float32).view(len(anchors), -1, 2)
    p[f"model.{det['i']}.anchors"] = a / torch.tensor(strides).view(-1, 1, 1)  # grid units, models/yolo.py:224
    for j, (c1, s) in enumerate(zip(chs, strides)):
        bound = 1.0 / math.sqrt(c1)
        p[f"model.{det['i']}.m.{j}.weight"] = (torch.rand(na * no, c1, 1, 1, generator=g) * 2 - 1) * bound
        b = ((torch.rand(na * no, generator=g) * 2 - 1) * bound).view(na, no)
        b[:, 4] += math.log(8 / (640 / s) ** 2)
        b[:, 5 : 5 + nc] += math.log(0.6 / (nc - 0.99999))
        p[f"model.{det['i']}.m.{j}.bias"] = b.view(-1)
    return p


def confident_params(cfg, seed=0):
    """``init_params`` with the objectness / class biases raised so that detections exist at ordinary thresholds (the
    shipped init gives conf ~ 3e-5 everywhere: nothing to compare)."""
    p = init_params(cfg, seed=seed)
    for k in p:
        if ".m." in k and k.endswith(".bias"):
            b = p[k].view(3, -1)
            b[:, 4] += 7.0   # sigmoid(-3.9 .. -5.3 + 7) = 0.85 .. 0.96
            b[:, 5:] += 5.0  # sigmoid(-4.9 + 5 +- noise) ~ 0.5: obj * cls crosses 0.25 for a share of the classes
    return p


def fold_bn(w, gamma, beta, mean, var, eps=BN_EPS):
    """fuse_conv_and_bn (ultralytics; semantic of models/yolo.py:163-172): W'=diag(g/sqrt(var+eps))W, b'=beta-g*mean/sqrt(var+eps)."""
    scale = gamma / torch.sqrt(var + eps)
    return w * scale.view(-1, 1, 1, 1), beta - mean * scale


# ----------------------------------------------------------------------------------------------------------------------
# Forward (models/yolo.py:135-147 executor semantics; models/common.py blocks; Detect models/yolo.py:89-123)
# ----------------------------------------------------------------------------------------------------------------------
class OracleModel:
    def __init__(self, cfg, params=None, seed=0, ch=3, fused=True, act_dtype=None, weight_dtype=None, train=False):
        """act_dtype/weight_dtype = torch.bfloat16 emulates the CUDA path's storage rounding (activations rounded to
        bf16 after every conv block, folded weights rounded to bf16, fp32 accumulation) for tight per-layer checks."""
        self.cfg = load_cfg(cfg)
        self.nodes, self.save = parse_graph(self.cfg, ch)
        self.params = params if params is not None else init_params(self.cfg, seed, ch=ch)
        self.fused = fused and not train
        self.train = train  # BatchNorm with batch statistics (train.py:403 runs the model in train mode)
        self.act_dtype, self.weight_dtype = act_dtype, weight_dtype
        det = self.nodes[-1]
        self.nc, anchors, _ = det["args"]
        self.nl, self.na, self.no = len(anchors), len(anchors[0]) // 2, self.nc + 5
        self.stride = torch.tensor(detect_strides(self.nodes, ch))
        self.anchors = self.params[f"model.{det['i']}.anchors"]  # grid units
        self.det_i = det["i"]

    def _round(self, x):
        return x.to(self.act_dtype).float() if self.act_dtype is not None else x

    def conv_block(self, x, prefix, k, s):
        """Conv.forward / forward_fuse, models/common.py:71-81: SiLU(BN(conv(x))), pad=k//2, bias=False."""
        P = self.params
        w = P[prefix + ".conv.weight"]
        bn = [P[prefix + ".bn." + n] for n in ("weight", "bias", "running_mean", "running_var")]
        if self.fused:
            w, b = fold_bn(w, *bn)
            if self.weight_dtype is not None:
                w = w.to(self.weight_dtype).float()
            y = F.conv2d(x, w, b, stride=s, padding=k // 2)
        elif self.train:
            y = F.conv2d(x, w, None, stride=s, padding=k // 2)
            y = F.batch_norm(y, None, None, bn[0], bn[1], True, 0.03, BN_EPS)
        else:
            y = F.conv2d(x, w, None, stride=s, padding=k // 2)
            y = F.batch_norm(y, bn[2], bn[3], bn[0], bn[1], False, 0.0, BN_EPS)
        return y * torch.sigmoid(y)

    def bottleneck(self, x, prefix, c1, c2, shortcut):
        """Bottleneck.forward, models/common.py:163-165."""
        y = self._round(self.conv_block(x, prefix + ".cv1", 1, 1))
        y = self.conv_block(y, prefix + ".cv2", 3, 1)
        return self._round(x + y if (shortcut and c1 == c2) else y)

    def forward_features(self, x, taps=None):
        """_forward_once, models/yolo.py:135-147.  Returns the list fed to Detect; fills ``taps`` {layer: tensor}."""
        y = []
        x = self._round(x)  # layer 0 of the CUDA path feeds bf16 MMAs: the image itself is rounded to bf16
        for nd in self.nodes:
            i, f, t = nd["i"], nd["f"], nd["type"]
            if t == "Detect":
                return [y[j] for j in f]
            if f != -1:
                x = y[f] if isinstance(f, int) else [x if j == -1 else y[j] for j in f]
            base = f"model.{i}"
            reps = [base] if nd["n"] == 1 else [f"{base}.{j}" for j in range(nd["n"])]
            if t == "Conv":
                c1, c2, *rest = nd["args"]
                k = rest[0] if len(rest) > 0 else 1
                s = rest[1] if len(rest) > 1 else 1
                for r in reps:
                    x = self._round(self.conv_block(x, r, k, s))
            elif t == "Bottleneck":
                c1, c2, *rest = nd["args"]
                shortcut = rest[0] if rest else True
                for r in reps:
                    x = self.bottleneck(x, r, c1, c2, shortcut)
                    c1 = c2
            elif t == "SPP":  # models/common.py:281-290
                c1, c2, *rest = nd["args"]
                ks = rest[0] if rest else (5, 9, 13)
                x = self._round(self.conv_block(x, base + ".cv1", 1, 1))
                x = torch.cat([x] + [F.max_pool2d(x, k, 1, k // 2) for k in ks], 1)
                x = self._round(self.conv_block(x, base + ".cv2", 1, 1))
            elif t == "MaxPool2d":
                k = nd["args"][0]
                s = nd["args"][1] if len(nd["args"]) > 1 else k
                pd = nd["args"][2] if len(nd["args"]) > 2 else 0
                x = F.max_pool2d(x, k, s, pd)
            elif t == "ZeroPad2d":
                x = F.pad(x, nd["args"][0])
            elif t == "Upsample":
                x = F.interpolate(x, scale_factor=nd["args"][1], mode=nd["args"][2])
            elif t == "Concat":
                x = torch.cat(x, nd["args"][0])
            y.append(x if i in self.save else None)
            if taps is not None and i in taps:
                taps[i] = x
        raise ValueError("graph has no Detect")

    def detect_raw(self, feats):
        """Detect.m[i] + view/permute, models/yolo.py:96-98 -> list of [bs,na,ny,nx,no] raw logits."""
        out = []
        for j, x in enumerate(feats):
            w = self.params[f"model.{self.det_i}.m.{j}.weight"]
            b = self.params[f"model.{self.det_i}.m.{j}.bias"]
            if self.weight_dtype is not None:
                w = w.to(self.weight_dtype).float()
            x = F.conv2d(x, w, b)
            bs, _, ny, nx = x.shape
            out.append(x.view(bs, self.na, self.no, ny, nx).permute(0, 1, 3, 4, 2).contiguous())
        return out

    def decode(self, raw):
        """Detect eval branch, models/yolo.py:100-108 + _make_grid :112-123 -> z[bs, sum(na*ny*nx), no]."""
        return decode(raw, self.anchors, self.stride)

    def forward(self, x, taps=None):
        """Eval-mode Model.forward: (z, [p_i]) as models/yolo.py:110."""
        raw = self.detect_raw(self.forward_features(x, taps))
        return self.decode(raw), raw

    __call__ = forward


def decode(raw, anchors_grid, stride):
    z = []
    for i, p in enumerate(raw):
        bs, na, ny, nx, no = p.shape
        yv, xv = torch.meshgrid(torch.arange(ny, dtype=torch.float32), torch.arange(nx, dtype=torch.float32), indexing="ij")
        grid = torch.stack((xv, yv), 2).expand(1, na, ny, nx, 2) - 0.5
        anchor_grid = (anchors_grid[i] * stride[i]).view(1, na, 1, 1, 2).expand(1, na, ny, nx, 2)
        s = p.float().sigmoid()
        xy = (s[..., 0:2] * 2 + grid) * stride[i]
        wh = (s[..., 2:4] * 2) ** 2 * anchor_grid
        z.append(torch.cat((xy, wh, s[..., 4:]), 4).view(bs, na * ny * nx, no))
    return torch.cat(z, 1)


# ----------------------------------------------------------------------------------------------------------------------
# NMS (utils/general.py:630-750 + torchvision.ops.nms).  numpy float32, no FMA contraction: every product/sum is a
# separately rounded fp32 op exactly as ATen's CPU kernels evaluate them.
# ----------------------------------------------------------------------------------------------------------------------
MAX_WH = np.float32(7680)  # utils/general.py:673
MAX_NMS = 30000  # utils/general.py:674


def greedy_nms(boxes, scores, iou_thres):
    """torchvision.ops.nms (CPU kernel semantics): stable descending score sort; keep i, suppress j>i iff
    inter/(area_i+area_j-inter) > thr (strict); area=(x2-x1)*(y2-y1); 0/0 -> NaN -> not suppressed."""
    boxes = np.asarray(boxes, dtype=np.float32)
    n = boxes.shape[0]
    if n == 0:
        return np.zeros((0,), dtype=np.int64)
    order = np.argsort(-np.asarray(scores, dtype=np.float32), kind="stable")
    b = boxes[order]
    x1, y1, x2, y2 = b[:, 0], b[:, 1], b[:, 2], b[:, 3]
    areas = ((x2 - x1) * (y2 - y1)).astype(np.float32)
    supp = np.zeros(n, dtype=bool)
    keep = []
    thr = np.float32(iou_thres)
    with np.errstate(divide="ignore", invalid="ignore"):
        for i in range(n):
            if supp[i]:
                continue
            keep.append(i)
            if i + 1 == n:
                break
            xx1 = np.maximum(x1[i], x1[i + 1 :])
            yy1 = np.maximum(y1[i], y1[i + 1 :])
            xx2 = np.minimum(x2[i], x2[i + 1 :])
            yy2 = np.minimum(y2[i], y2[i + 1 :])
            w = np.maximum(np.float32(0), (xx2 - xx1).astype(np.float32))
            h = np.maximum(np.float32(0), (yy2 - yy1).astype(np.float32))
            inter = (w * h).astype(np.float32)
            union = ((areas[i] + areas[i + 1 :]).astype(np.float32) - inter).astype(np.float32)
            ovr = (inter / union).astype(np.float32)
            supp[i + 1 :] |= ovr > thr
    return order[np.asarray(keep, dtype=np.int64)]


def nms_image(x, conf_thres=0.25, iou_thres=0.45, classes=None, agnostic=False, multi_label=False, max_det=300, lb=None,
              use_torchvision=False):
    """One image of non_max_suppression (utils/general.py:683-743).  x: [n, 5+nc] float32.

    Returns (det[k,6] float32 = xyxy,conf,cls sorted by conf desc; src[k,2] int64 = (row, cls) of each kept detection).
    Ties in conf are broken by candidate order (row-major (row, cls)), i.e. a *stable* descending sort; the
    reference's ``argsort(descending=True)`` (:728) is unstable, so parity on tied scores is only defined up to the
    tie group (SURVEY App. C.3) and the goldens are tie-free.
    """
    x = np.asarray(x, dtype=np.float32)
    nc = x.shape[1] - 5
    n_pred = x.shape[0]
    multi_label = multi_label and nc > 1
    thr = np.float32(conf_thres)
    rows = np.nonzero(x[:, 4] > thr)[0]  # :669,686
    x = x[rows]
    if lb is not None and len(lb):  # autolabel priors appended AFTER the confidence filter (:689-695); src row = n + i
        lb = np.asarray(lb, dtype=np.float32).reshape(-1, 5)
        v = np.zeros((len(lb), nc + 5), np.float32)
        v[:, :4] = lb[:, 1:5]
        v[:, 4] = 1.0
        v[np.arange(len(lb)), lb[:, 0].astype(np.int64) + 5] = 1.0
        rows = np.concatenate((rows, np.arange(len(lb)) + n_pred))
        x = np.concatenate((x, v), 0)
    empty = (np.zeros((0, 6), np.float32), np.zeros((0, 2), np.int64))
    if x.shape[0] == 0:
        return empty
    conf_all = (x[:, 5:] * x[:, 4:5]).astype(np.float32)  # :702
    half = (x[:, 2:4] / np.float32(2)).astype(np.float32)  # xywh2xyxy :705
    box = np.concatenate(((x[:, 0:2] - half).astype(np.float32), (x[:, 0:2] + half).astype(np.float32)), 1)
    if multi_label:  # :710-711
        i, j = np.nonzero(conf_all > thr)
        det = np.concatenate((box[i], conf_all[i, j, None], j[:, None].astype(np.float32)), 1)
        src = np.stack((rows[i], j), 1)
    else:  # :713-714
        j = conf_all.argmax(1)
        conf = conf_all[np.arange(len(j)), j]
        m = conf > thr
        det = np.concatenate((box, conf[:, None], j[:, None].astype(np.float32)), 1)[m]
        src = np.stack((rows, j), 1)[m]
    if classes is not None:  # :717-718
        m = np.isin(det[:, 5].astype(np.int64), np.asarray(classes, dtype=np.int64))
        det, src = det[m], src[m]
    if det.shape[0] == 0:
        return empty
    order = np.argsort(-det[:, 4], kind="stable")[:MAX_NMS]  # :728
    det, src = det[order], src[order]
    c = (det[:, 5:6] * (np.float32(0) if agnostic else MAX_WH)).astype(np.float32)  # :731
    boxes = (det[:, :4] + c).astype(np.float32)  # :732
    if use_torchvision:  # the reference's own call (general.py:733); same kept set as greedy_nms on tie-free scores
        import torchvision

        keep = torchvision.ops.nms(torch.from_numpy(boxes), torch.from_numpy(np.ascontiguousarray(det[:, 4])), iou_thres).numpy()[:max_det]
    else:
        keep = greedy_nms(boxes, det[:, 4], iou_thres)[:max_det]  # :733-734
    return det[keep].astype(np.float32), src[keep].astype(np.int64)


def non_max_suppression(prediction, conf_thres=0.25, iou_thres=0.45, classes=None, agnostic=False, multi_label=False,
                        max_det=300, labels=(), use_torchvision=False):
    """Batch wrapper; the reference's wall-clock ``time_limit`` break (utils/general.py:675,746-748) is NOT restated:
    it is a hazard, not a result (SURVEY App. C.1)."""
    assert 0 <= conf_thres <= 1 and 0 <= iou_thres <= 1
    if isinstance(prediction, (list, tuple)):
        prediction = prediction[0]
    pred = prediction.detach().cpu().float().numpy() if isinstance(prediction, torch.Tensor) else np.asarray(prediction)
    outs, srcs = [], []
    for xi in range(pred.shape[0]):
        d, s = nms_image(pred[xi], conf_thres, iou_thres, classes, agnostic, multi_label, max_det,
                         lb=labels[xi] if labels else None, use_torchvision=use_torchvision)
        outs.append(d)
        srcs.append(s)
    return outs, srcs


def scale_boxes(img1_shape, boxes, img0_shape, ratio_pad=None):
    """utils/general.py:613-626 (+ ultralytics clip_boxes): un-letterbox xyxy boxes and clip them; numpy float32, every
    step separately rounded like the torch ops (tensor -= python float, tensor /= python float, clamp)."""
    b = np.array(boxes, dtype=np.float32, copy=True)
    if ratio_pad is None:
        gain = min(img1_shape[0] / img0_shape[0], img1_shape[1] / img0_shape[1])
        pad = (img1_shape[1] - img0_shape[1] * gain) / 2, (img1_shape[0] - img0_shape[0] * gain) / 2
    else:
        gain, pad = ratio_pad[0][0], ratio_pad[1]
    b[..., [0, 2]] = (b[..., [0, 2]] - np.float32(pad[0])).astype(np.float32)
    b[..., [1, 3]] = (b[..., [1, 3]] - np.float32(pad[1])).astype(np.float32)
    b[..., :4] = (b[..., :4] / np.float32(gain)).astype(np.float32)
    b[..., [0, 2]] = np.clip(b[..., [0, 2]], np.float32(0), np.float32(img0_shape[1]))
    b[..., [1, 3]] = np.clip(b[..., [1, 3]], np.float32(0), np.float32(img0_shape[0]))
    return b


# ------------------------------------------------------------------------------------------------ TTA
def scale_img(img, ratio=1.0, same_shape=False, gs=32):
    """ultralytics scale_img (third-party; used by models/yolo.py:246): bilinear resize to int(h*r) x int(w*r), right/bottom pad
    with 0.447 to a gs multiple."""
    if ratio == 1.0:
        return img
    h, w = img.shape[2:]
    s = (int(h * ratio), int(w * ratio))
    img = F.interpolate(img, size=s, mode="bilinear", align_corners=False)
    if not same_shape:
        h, w = (math.ceil(x * ratio / gs) * gs for x in (h, w))
    return F.pad(img, [0, w - s[1], 0, h - s[0]], value=0.447)


def forward_augment(om, x):
    """Model._forward_augment + _descale_pred + _clip_augmented (models/yolo.py:239-278) on an OracleModel: returns z_aug."""
    img_size = x.shape[-2:]
    y = []
    for si, fi in zip([1, 0.83, 0.67], [None, 3, None]):
        xi = scale_img(x.flip(fi) if fi else x, si, gs=int(max(om.stride)))
        yi = om(xi)[0].clone()
        yi[..., :4] /= si
        if fi == 3:
            yi[..., 0] = img_size[1] - yi[..., 0]
        y.append(yi)
    nl = len(om.stride)
    g = sum(4 ** q for q in range(nl))
    i = (y[0].shape[1] // g) * 1
    y[0] = y[0][:, :-i]
    i = (y[-1].shape[1] // g) * 4 ** (nl - 1)
    y[-1] = y[-1][:, i:]
    return torch.cat(y, 1)


# ------------------------------------------------------------------------------------------------ pre-processing
def _cv_round(x):
    """cvRound / saturate_cast<short>(float): round half to even."""
    return np.rint(x).astype(np.int64)


def resize_linear_u8(src, dw, dh):
    """cv2.resize(src, (dw, dh), interpolation=cv2.INTER_LINEAR) for uint8 HWC images, restated bit-exactly from OpenCV's
    fixed-point path (third-party: opencv-python 4.13 is what the reference's letterbox calls, utils/augmentations.py:127;
    resize.cpp: 11-bit coefficients, HResizeLinear -> int, VResizeLinear ((b*(S>>4))>>16 ... +2)>>2; the exact 2x shrink takes
    the INTER_AREA 2x2 average).  Pinned against cv2 itself in tests/test_oracle_golden.py."""
    sh, sw = src.shape[:2]
    if (dw, dh) == (sw, sh):
        return src.copy()
    scale_x, scale_y = 1.0 / (dw / sw), 1.0 / (dh / sh)
    isx, isy = int(np.rint(scale_x)), int(np.rint(scale_y))
    eps = np.finfo(np.float64).eps
    if abs(scale_x - isx) < eps and abs(scale_y - isy) < eps and isx == 2 and isy == 2:
        s = src.astype(np.int32)
        return ((s[0:2 * dh:2, 0:2 * dw:2] + s[0:2 * dh:2, 1:2 * dw:2] + s[1:2 * dh:2, 0:2 * dw:2] + s[1:2 * dh:2, 1:2 * dw:2] + 2)
                >> 2).astype(np.uint8)

    def frac(dn, scale):
        f = ((np.arange(dn) + 0.5) * scale - 0.5).astype(np.float32)
        s0 = np.floor(f).astype(np.int64)
        return s0, (f - s0.astype(np.float32)).astype(np.float32)

    sx, fx = frac(dw, scale_x)
    lo, hi = sx < 0, sx >= sw - 1
    fx[lo], sx[lo] = 0, 0
    fx[hi], sx[hi] = 0, sw - 1
    ax0, ax1 = _cv_round((np.float32(1.0) - fx) * np.float32(2048)), _cv_round(fx * np.float32(2048))
    sy, fy = frac(dh, scale_y)
    b0, b1 = _cv_round((np.float32(1.0) - fy) * np.float32(2048)), _cv_round(fy * np.float32(2048))
    s = src.astype(np.int64)
    hrow = s[:, sx] * ax0[None, :, None] + s[:, np.minimum(sx + 1, sw - 1)] * ax1[None, :, None]
    s0, s1 = hrow[np.clip(sy, 0, sh - 1)], hrow[np.clip(sy + 1, 0, sh - 1)]
    out = (((b0[:, None, None] * (s0 >> 4)) >> 16) + ((b1[:, None, None] * (s1 >> 4)) >> 16) + 2) >> 2
    return out.astype(np.uint8)


def letterbox_geometry(shape, new_shape=(640, 640), auto=True, scaleFill=False, scaleup=True, stride=32):
    """The scalar part of letterbox (utils/augmentations.py:104-132): returns (new_unpad (w, h), ratio, (dw, dh), top, bottom,
    left, right)."""
    if isinstance(new_shape, int):
        new_shape = (new_shape, new_shape)
    r = min(new_shape[0] / shape[0], new_shape[1] / shape[1])
    if not scaleup:
        r = min(r, 1.0)
    ratio = r, r
    new_unpad = round(shape[1] * r), round(shape[0] * r)
    dw, dh = new_shape[1] - new_unpad[0], new_shape[0] - new_unpad[1]
    if auto:
        dw, dh = np.mod(dw, stride), np.mod(dh, stride)
    elif scaleFill:
        dw, dh = 0.0, 0.0
        new_unpad = (new_shape[1], new_shape[0])
        ratio = new_shape[1] / shape[1], new_shape[0] / shape[0]
    dw /= 2
    dh /= 2
    top, bottom = round(dh - 0.1), round(dh + 0.1)
    left, right = round(dw - 0.1), round(dw + 0.1)
    return new_unpad, ratio, (dw, dh), top, bottom, left, right


def letterbox(im, new_shape=(640, 640), color=(114, 114, 114), auto=True, scaleFill=False, scaleup=True, stride=32):
    """letterbox (utils/augmentations.py:104-134) on a uint8 HWC numpy image: cv2.resize(INTER_LINEAR) + constant border."""
    new_unpad, ratio, (dw, dh), top, bottom, left, right = letterbox_geometry(im.shape[:2], new_shape, auto, scaleFill, scaleup, stride)
    if im.shape[:2][::-1] != new_unpad:
        im = resize_linear_u8(im, new_unpad[0], new_unpad[1])
    out = np.empty((im.shape[0] + top + bottom, im.shape[1] + left + right, im.shape[2]), np.uint8)
    out[...] = np.asarray(color, np.uint8)
    out[top:top + im.shape[0], left:left + im.shape[1]] = im
    return out, ratio, (dw, dh)


def preprocess(im0, img_size=640, stride=32, auto=True):
    """LoadImages.__next__ (utils/dataloaders.py:305-310): letterbox -> HWC to CHW, BGR to RGB -> contiguous uint8."""
    im = letterbox(im0, img_size, stride=stride, auto=auto)[0]
    return np.ascontiguousarray(im.transpose((2, 0, 1))[::-1])


def process_batch(detections, labels, iouv):
    """val.process_batch (reference val.py:147-188) restated with the same torch / numpy calls in the same order:
    detections [N,6] (xyxy, conf, cls), labels [M,5] (cls, xyxy), iouv [T] -> bool [N,T]."""
    correct = np.zeros((detections.shape[0], iouv.shape[0])).astype(bool)
    iou = box_iou(labels[:, 1:], detections[:, :4])
    correct_class = labels[:, 0:1] == detections[:, 5]
    for i in range(len(iouv)):
        x = torch.where((iou >= iouv[i]) & correct_class)  # val.py:179
        if x[0].shape[0]:
            matches = torch.cat((torch.stack(x, 1), iou[x[0], x[1]][:, None]), 1).cpu().numpy()  # [label, detect, iou]
            if x[0].shape[0] > 1:
                matches = matches[matches[:, 2].argsort()[::-1]]
                matches = matches[np.unique(matches[:, 1], return_index=True)[1]]
                matches = matches[np.unique(matches[:, 0], return_index=True)[1]]
            correct[matches[:, 1].astype(int), i] = True
    return torch.tensor(correct, dtype=torch.bool)


def synth_val_case(n_det=120, n_lab=25, nc=6, seed=0, jitter=12.0, size=640.0):
    """Seeded detections/labels for the matching tests: labels are random boxes, most detections are jittered copies of a
    label (several per label, some with the wrong class), the rest random; detections sorted by confidence like NMS output."""
    g = torch.Generator().manual_seed(seed)
    xy = torch.rand(n_lab, 2, generator=g) * (size - 200) + 20
    wh = torch.rand(n_lab, 2, generator=g) * 160 + 20
    lab = torch.cat((torch.randint(0, nc, (n_lab, 1), generator=g).float(), xy, xy + wh), 1)
    src = torch.randint(0, max(n_lab, 1), (n_det,), generator=g)
    box = lab[src, 1:] + torch.randn(n_det, 4, generator=g) * jitter if n_lab else torch.zeros(n_det, 4)
    rnd = torch.rand(n_det, generator=g) < 0.2
    rxy = torch.rand(n_det, 2, generator=g) * (size - 100)
    box[rnd] = torch.cat((rxy, rxy + torch.rand(n_det, 2, generator=g) * 90 + 10), 1)[rnd]
    cls = lab[src, 0].clone() if n_lab else torch.zeros(n_det)
    wrong = torch.rand(n_det, generator=g) < 0.15
    cls[wrong] = torch.randint(0, nc, (int(wrong.sum()),), generator=g).float()
    conf = torch.rand(n_det, generator=g).sort(descending=True).values
    det = torch.cat((box, conf[:, None], cls[:, None]), 1)
    return det, lab


def box_iou(box1, box2, eps=1e-7):
    """ultralytics box_iou (re-exported utils/metrics.py:10; used val.py:176): inter/(a1+a2-inter+eps), [N,M]."""
    b1, b2 = torch.as_tensor(box1).float(), torch.as_tensor(box2).float()
    lt = torch.max(b1[:, None, :2], b2[None, :, :2])
    rb = torch.min(b1[:, None, 2:], b2[None, :, 2:])
    inter = (rb - lt).clamp(min=0).prod(2)
    a1 = (b1[:, 2] - b1[:, 0]) * (b1[:, 3] - b1[:, 1])
    a2 = (b2[:, 2] - b2[:, 0]) * (b2[:, 3] - b2[:, 1])
    return inter / (a1[:, None] + a2[None, :] - inter + eps)


# ----------------------------------------------------------------------------------------------------------------------
# Loss (utils/loss.py:98-244 + ultralytics bbox_iou(CIoU), smooth_bce).  torch CPU fp32; autograd supplies dL/dp.
# ----------------------------------------------------------------------------------------------------------------------
def ciou_xywh(b1, b2, eps=1e-7):
    """bbox_iou(box1, box2, xywh=True, CIoU=True) (ultralytics; called utils/loss.py:151).  [n,4]x[n,4]->[n]."""
    x1, y1, w1, h1 = b1.unbind(-1)
    x2, y2, w2, h2 = b2.unbind(-1)
    b1x1, b1x2, b1y1, b1y2 = x1 - w1 / 2, x1 + w1 / 2, y1 - h1 / 2, y1 + h1 / 2
    b2x1, b2x2, b2y1, b2y2 = x2 - w2 / 2, x2 + w2 / 2, y2 - h2 / 2, y2 + h2 / 2
    inter = (torch.minimum(b1x2, b2x2) - torch.maximum(b1x1, b2x1)).clamp(0) * (
        torch.minimum(b1y2, b2y2) - torch.maximum(b1y1, b2y1)
    ).clamp(0)
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


DEFAULT_HYP = dict(box=0.05, obj=1.0, cls=0.5, cls_pw=1.0, obj_pw=1.0, fl_gamma=0.0, anchor_t=4.0,
                   label_smoothing=0.0)  # data/hyps/hyp.scratch-low.yaml values on the loss path


def scaled_hyp(hyp=None, nl=3, nc=80, imgsz=640):
    """train.py:326-329 rescale of box/cls/obj gains."""
    h = dict(DEFAULT_HYP if hyp is None else hyp)
    h["box"] *= 3 / nl
    h["cls"] *= nc / 80 * 3 / nl
    h["obj"] *= (imgsz / 640) ** 2 * 3 / nl
    return h


def build_targets(shapes, targets, anchors, anchor_t=4.0):
    """ComputeLoss.build_targets, utils/loss.py:183-244.  shapes: list of (bs,na,ny,nx,no); targets [nt,6]
    (img,cls,x,y,w,h normalised); anchors [nl,na,2] grid units.  Returns per level (b,a,gj,gi,tbox[n,4],anch[n,2],tcls)."""
    targets = torch.as_tensor(targets, dtype=torch.float32)
    na, nt = anchors.shape[1], targets.shape[0]
    out = []
    g = 0.5
    off = torch.tensor([[0, 0], [1, 0], [0, 1], [-1, 0], [0, -1]], dtype=torch.float32) * g
    for i, shape in enumerate(shapes):
        ny, nx = shape[2], shape[3]
        gain = torch.tensor([1, 1, nx, ny, nx, ny, 1], dtype=torch.float32)
        ai = torch.arange(na, dtype=torch.float32).view(na, 1).repeat(1, nt)
        t = torch.cat((targets.repeat(na, 1, 1), ai[..., None]), 2) * gain  # [na,nt,7]
        if nt:
            r = t[..., 4:6] / anchors[i][:, None]
            j = torch.max(r, 1 / r).max(2)[0] < anchor_t
            t = t[j]
            gxy = t[:, 2:4]
            gxi = gain[[2, 3]] - gxy
            jj, kk = ((gxy % 1 < g) & (gxy > 1)).T
            ll, mm = ((gxi % 1 < g) & (gxi > 1)).T
            sel = torch.stack((torch.ones_like(jj), jj, kk, ll, mm))
            t = t.repeat((5, 1, 1))[sel]
            offsets = (torch.zeros_like(gxy)[None] + off[:, None])[sel]
        else:
            t = t[0]
            offsets = 0
        b, c = t[:, 0].long(), t[:, 1].long()
        gxy, gwh, a = t[:, 2:4], t[:, 4:6], t[:, 6].long()
        gij = (gxy - offsets).long()
        gi, gj = gij[:, 0].clamp(0, nx - 1), gij[:, 1].clamp(0, ny - 1)
        # the reference's gi, gj are views of gij and are clamped in place (loss.py:236-239) one statement before tbox is
        # formed (:240), so tbox uses the CLAMPED indices: a centre at x = 1.0 gives tx = 1.0 in cell nx - 1, not 0.0
        gij = torch.stack((gi, gj), 1)
        out.append(dict(b=b, a=a, gj=gj, gi=gi, tbox=torch.cat((gxy - gij, gwh), 1), anch=anchors[i][a], tcls=c))
    return out


def compute_loss(p, targets, anchors, hyp, nc=80):
    """ComputeLoss.__call__, utils/loss.py:131-181 (fl_gamma=0, autobalance off, gr=1).  p: list of raw [bs,na,ny,nx,no]
    (requires_grad for dL/dp).  Returns (loss[1], loss_items[3]=(lbox,lobj,lcls))."""
    nl = len(p)
    balance = {3: [4.0, 1.0, 0.4]}.get(nl, [4.0, 1.0, 0.25, 0.06, 0.02])
    cp, cn = 1.0 - 0.5 * hyp.get("label_smoothing", 0.0), 0.5 * hyp.get("label_smoothing", 0.0)
    tg = build_targets([tuple(pi.shape) for pi in p], targets, anchors, hyp["anchor_t"])
    lcls, lbox, lobj = torch.zeros(1), torch.zeros(1), torch.zeros(1)
    cls_pw, obj_pw = torch.tensor([hyp["cls_pw"]]), torch.tensor([hyp["obj_pw"]])
    for i, pi in enumerate(p):
        t = tg[i]
        b, a, gj, gi = t["b"], t["a"], t["gj"], t["gi"]
        tobj = torch.zeros(pi.shape[:4], dtype=pi.dtype)
        n = b.shape[0]
        if n:
            ps = pi[b, a, gj, gi]
            pxy = ps[:, 0:2].sigmoid() * 2 - 0.5
            pwh = (ps[:, 2:4].sigmoid() * 2) ** 2 * t["anch"]
            iou = ciou_xywh(torch.cat((pxy, pwh), 1), t["tbox"])
            lbox = lbox + (1.0 - iou).mean()
            tobj[b, a, gj, gi] = iou.detach().clamp(0).type(tobj.dtype)  # last-write-wins on duplicates (:161)
            if nc > 1:
                tc = torch.full_like(ps[:, 5:], cn)
                tc[range(n), t["tcls"]] = cp
                lcls = lcls + F.binary_cross_entropy_with_logits(ps[:, 5:], tc, pos_weight=cls_pw)
        lobj = lobj + F.binary_cross_entropy_with_logits(pi[..., 4], tobj, pos_weight=obj_pw) * balance[i]
    lbox, lobj, lcls = lbox * hyp["box"], lobj * hyp["obj"], lcls * hyp["cls"]
    bs = p[0].shape[0]
    return (lbox + lobj + lcls) * bs, torch.cat((lbox, lobj, lcls)).detach()


# ----------------------------------------------------------------------------------------------------------------------
# Synthetic workloads (SURVEY §8(d)): shared by tests and bench so every arm sees the same inputs
# ----------------------------------------------------------------------------------------------------------------------
def synth_predictions(bs, n_rows=25200, nc=80, seed=3, imgsz=640):
    """Config 5 NMS input: xy~U(0,imgsz), wh~U(4,204), obj~U(0,1)^6, cls~U(0,1)^4."""
    g = torch.Generator().manual_seed(seed)
    p = torch.empty(bs, n_rows, 5 + nc)
    p[..., 0:2] = torch.rand(bs, n_rows, 2, generator=g) * imgsz
    p[..., 2:4] = torch.rand(bs, n_rows, 2, generator=g) * 200 + 4
    p[..., 4] = torch.rand(bs, n_rows, generator=g) ** 6
    p[..., 5:] = torch.rand(bs, n_rows, nc, generator=g) ** 4
    return p


def synth_targets(bs, nc=80, seed=2):
    """Config 4 targets, coco128-shaped: n~Poisson(7.3) clipped [1,40]/img, cls~U{0..nc-1}, xy~U(.05,.95),
    wh~LogUniform(.02,.6) clipped inside the image; layout [nt,6]=(img,cls,x,y,w,h) as collate_fn
    (utils/dataloaders.py:825-830)."""
    g = torch.Generator().manual_seed(seed)
    rows = []
    for b in range(bs):
        n = int(torch.poisson(torch.tensor(7.3), generator=g).clamp(1, 40))
        cls = torch.randint(0, nc, (n,), generator=g).float()
        xy = torch.rand(n, 2, generator=g) * 0.9 + 0.05
        wh = torch.exp(torch.rand(n, 2, generator=g) * (math.log(0.6) - math.log(0.02)) + math.log(0.02))
        wh = torch.minimum(wh, 2 * torch.minimum(xy, 1 - xy))
        rows.append(torch.cat((torch.full((n, 1), float(b)), cls[:, None], xy, wh), 1))
    return torch.cat(rows, 0)

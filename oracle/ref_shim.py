"""TEST INFRASTRUCTURE ONLY — import shim for running the *reference* (``/root/reference``) in the build container.

The reference imports ``ultralytics>=8.4.110`` (requirements.txt:18, pyproject.toml:78), ``matplotlib`` and ``seaborn``;
none of them is installed here and there is no network.  This module registers in-memory stand-ins for exactly the symbols
the reference imports (utils/general.py:32-55, utils/torch_utils.py:13-21, utils/loss.py:6, utils/metrics.py:10,
utils/__init__.py:6, models/common.py, models/experimental.py, utils/plots.py, utils/dataloaders.py,
utils/augmentations.py) so that the reference files import UNMODIFIED.  The arithmetic symbols (``bbox_iou``, ``box_iou``,
``fuse_conv_and_bn``, ``xywh2xyxy`` ...) are third-party code that is absent from ``/root/reference``; they are restated
here from the published ultralytics 8.x formulas (SURVEY.md Appendix B) and unit-tested independently in
``tests/golden/make_golden.py`` (``gen_iou``: float64 CIoU cross-check, ``torchvision.ops.box_iou``; ``gen_forward``: fused
vs unfused forward through ``fuse_conv_and_bn``) and re-checked from the fixtures by ``tests/test_oracle_golden.py``.

Consumers: ``tests/golden/make_golden.py`` (golden-vector generation, pointed at a checkout of the reference with
``--reference``) and ``bench.py``'s reference legs, which run the byte-for-byte copy that ``build()`` stages under the
git-ignored ``oracle/_ref/`` (``oracle/stage_reference.py``) when a reference checkout is at hand.  No test reads the
reference: what they compare against is stored under ``tests/golden/``.  Nothing under ``yolov3_b200/`` imports this.
"""
from __future__ import annotations

import contextlib
import logging
import math
import sys
import time
import types
from copy import deepcopy
from pathlib import Path

import torch
import torch.nn as nn

_REPO = Path(__file__).resolve().parents[1]
# the copy build() stages (oracle/stage_reference.py); make_golden.py points this at a reference checkout instead
REFERENCE_ROOT = _REPO / "oracle" / "_ref"


# ----------------------------------------------------------------------------------------------------------------------
# ultralytics.utils.ops
# ----------------------------------------------------------------------------------------------------------------------
def make_divisible(x, divisor):
    if isinstance(divisor, torch.Tensor):
        divisor = int(divisor.max())
    return math.ceil(x / divisor) * divisor


def xywh2xyxy(x):
    y = torch.empty_like(x) if isinstance(x, torch.Tensor) else x.copy()
    xy = x[..., :2]
    wh = x[..., 2:] / 2
    y[..., :2] = xy - wh
    y[..., 2:] = xy + wh
    return y


def xyxy2xywh(x):
    y = torch.empty_like(x) if isinstance(x, torch.Tensor) else x.copy()
    y[..., 0] = (x[..., 0] + x[..., 2]) / 2
    y[..., 1] = (x[..., 1] + x[..., 3]) / 2
    y[..., 2] = x[..., 2] - x[..., 0]
    y[..., 3] = x[..., 3] - x[..., 1]
    return y


def xywhn2xyxy(x, w=640, h=640, padw=0, padh=0):
    y = torch.empty_like(x) if isinstance(x, torch.Tensor) else x.copy()
    y[..., 0] = w * (x[..., 0] - x[..., 2] / 2) + padw
    y[..., 1] = h * (x[..., 1] - x[..., 3] / 2) + padh
    y[..., 2] = w * (x[..., 0] + x[..., 2] / 2) + padw
    y[..., 3] = h * (x[..., 1] + x[..., 3] / 2) + padh
    return y


def clip_boxes(boxes, shape):
    if isinstance(boxes, torch.Tensor):
        boxes[..., 0] = boxes[..., 0].clamp(0, shape[1])
        boxes[..., 1] = boxes[..., 1].clamp(0, shape[0])
        boxes[..., 2] = boxes[..., 2].clamp(0, shape[1])
        boxes[..., 3] = boxes[..., 3].clamp(0, shape[0])
    else:
        boxes[..., [0, 2]] = boxes[..., [0, 2]].clip(0, shape[1])
        boxes[..., [1, 3]] = boxes[..., [1, 3]].clip(0, shape[0])
    return boxes


def xyxy2xywhn(x, w=640, h=640, clip=False, eps=0.0):
    if clip:
        x = clip_boxes(x, (h - eps, w - eps))
    y = torch.empty_like(x) if isinstance(x, torch.Tensor) else x.copy()
    y[..., 0] = ((x[..., 0] + x[..., 2]) / 2) / w
    y[..., 1] = ((x[..., 1] + x[..., 3]) / 2) / h
    y[..., 2] = (x[..., 2] - x[..., 0]) / w
    y[..., 3] = (x[..., 3] - x[..., 1]) / h
    return y


class Profile(contextlib.ContextDecorator):
    def __init__(self, t=0.0, device=None):
        self.t = t
        self.dt = 0.0
        self.device = device
        self.cuda = bool(device and str(device).startswith("cuda"))

    def __enter__(self):
        self.start = self.time()
        return self

    def __exit__(self, *a):
        self.dt = self.time() - self.start
        self.t += self.dt

    def time(self):
        if self.cuda:
            torch.cuda.synchronize(self.device)
        return time.perf_counter()


# ----------------------------------------------------------------------------------------------------------------------
# ultralytics.utils.metrics
# ----------------------------------------------------------------------------------------------------------------------
def box_iou(box1, box2, eps=1e-7):
    (a1, a2), (b1, b2) = box1.float().unsqueeze(1).chunk(2, 2), box2.float().unsqueeze(0).chunk(2, 2)
    inter = (torch.min(a2, b2) - torch.max(a1, b1)).clamp_(0).prod(2)
    return inter / ((a2 - a1).prod(2) + (b2 - b1).prod(2) - inter + eps)


def bbox_iou(box1, box2, xywh=True, GIoU=False, DIoU=False, CIoU=False, eps=1e-7):
    if xywh:
        (x1, y1, w1, h1), (x2, y2, w2, h2) = box1.chunk(4, -1), box2.chunk(4, -1)
        w1_, h1_, w2_, h2_ = w1 / 2, h1 / 2, w2 / 2, h2 / 2
        b1_x1, b1_x2, b1_y1, b1_y2 = x1 - w1_, x1 + w1_, y1 - h1_, y1 + h1_
        b2_x1, b2_x2, b2_y1, b2_y2 = x2 - w2_, x2 + w2_, y2 - h2_, y2 + h2_
    else:
        b1_x1, b1_y1, b1_x2, b1_y2 = box1.chunk(4, -1)
        b2_x1, b2_y1, b2_x2, b2_y2 = box2.chunk(4, -1)
        w1, h1 = b1_x2 - b1_x1, b1_y2 - b1_y1 + eps
        w2, h2 = b2_x2 - b2_x1, b2_y2 - b2_y1 + eps
    inter = (b1_x2.minimum(b2_x2) - b1_x1.maximum(b2_x1)).clamp_(0) * (
        b1_y2.minimum(b2_y2) - b1_y1.maximum(b2_y1)
    ).clamp_(0)
    union = w1 * h1 + w2 * h2 - inter + eps
    iou = inter / union
    if CIoU or DIoU or GIoU:
        cw = b1_x2.maximum(b2_x2) - b1_x1.minimum(b2_x1)
        ch = b1_y2.maximum(b2_y2) - b1_y1.minimum(b2_y1)
        if CIoU or DIoU:
            c2 = cw.pow(2) + ch.pow(2) + eps
            rho2 = ((b2_x1 + b2_x2 - b1_x1 - b1_x2).pow(2) + (b2_y1 + b2_y2 - b1_y1 - b1_y2).pow(2)) / 4
            if CIoU:
                v = (4 / math.pi**2) * ((w2 / h2).atan() - (w1 / h1).atan()).pow(2)
                with torch.no_grad():
                    alpha = v / (v - iou + (1 + eps))
                return iou - (rho2 / c2 + v * alpha)
            return iou - rho2 / c2
        c_area = cw * ch + eps
        return iou - (c_area - union) / c_area
    return iou


def bbox_ioa(box1, box2, iou=False, eps=1e-7):
    import numpy as np

    b1_x1, b1_y1, b1_x2, b1_y2 = box1.T
    b2_x1, b2_y1, b2_x2, b2_y2 = box2.T
    inter_area = (np.minimum(b1_x2[:, None], b2_x2) - np.maximum(b1_x1[:, None], b2_x1)).clip(0) * (
        np.minimum(b1_y2[:, None], b2_y2) - np.maximum(b1_y1[:, None], b2_y1)
    ).clip(0)
    area = (b2_x2 - b2_x1) * (b2_y2 - b2_y1)
    if iou:
        box1_area = (b1_x2 - b1_x1) * (b1_y2 - b1_y1)
        area = area + box1_area[:, None] - inter_area
    return inter_area / (area + eps)


def smooth_bce(eps=0.1):
    return 1.0 - 0.5 * eps, 0.5 * eps


def smooth(y, f=0.05):
    import numpy as np

    nf = round(len(y) * f * 2) // 2 + 1
    p = np.ones(nf // 2)
    yp = np.concatenate((p * y[0], y, p * y[-1]), 0)
    return np.convolve(yp, np.ones(nf) / nf, mode="valid")


# ----------------------------------------------------------------------------------------------------------------------
# ultralytics.utils.torch_utils
# ----------------------------------------------------------------------------------------------------------------------
def fuse_conv_and_bn(conv, bn):
    fusedconv = (
        nn.Conv2d(
            conv.in_channels,
            conv.out_channels,
            kernel_size=conv.kernel_size,
            stride=conv.stride,
            padding=conv.padding,
            dilation=conv.dilation,
            groups=conv.groups,
            bias=True,
        )
        .requires_grad_(False)
        .to(conv.weight.device)
    )
    w_conv = conv.weight.view(conv.out_channels, -1)
    w_bn = torch.diag(bn.weight.div(torch.sqrt(bn.eps + bn.running_var)))
    fusedconv.weight.copy_(torch.mm(w_bn, w_conv).view(fusedconv.weight.shape))
    b_conv = torch.zeros(conv.weight.shape[0], device=conv.weight.device) if conv.bias is None else conv.bias
    b_bn = bn.bias - bn.weight.mul(bn.running_mean).div(torch.sqrt(bn.running_var + bn.eps))
    fusedconv.bias.copy_(torch.mm(w_bn, b_conv.reshape(-1, 1)).reshape(-1) + b_bn)
    return fusedconv


def initialize_weights(model):
    for m in model.modules():
        t = type(m)
        if t is nn.Conv2d:
            pass
        elif t is nn.BatchNorm2d:
            m.eps = 1e-3
            m.momentum = 0.03
        elif t in {nn.Hardswish, nn.LeakyReLU, nn.ReLU, nn.ReLU6, nn.SiLU}:
            m.inplace = True


def scale_img(img, ratio=1.0, same_shape=False, gs=32):
    import torch.nn.functional as F

    if ratio == 1.0:
        return img
    h, w = img.shape[2:]
    s = (int(h * ratio), int(w * ratio))
    img = F.interpolate(img, size=s, mode="bilinear", align_corners=False)
    if not same_shape:
        h, w = (math.ceil(x * ratio / gs) * gs for x in (h, w))
    return F.pad(img, [0, w - s[1], 0, h - s[0]], value=0.447)


def copy_attr(a, b, include=(), exclude=()):
    for k, v in b.__dict__.items():
        if (len(include) and k not in include) or k.startswith("_") or k in exclude:
            continue
        setattr(a, k, v)


class ModelEMA:
    def __init__(self, model, decay=0.9999, tau=2000, updates=0):
        self.ema = deepcopy(model.module if hasattr(model, "module") else model).eval()
        self.updates = updates
        self.decay = lambda x: decay * (1 - math.exp(-x / tau))
        for p in self.ema.parameters():
            p.requires_grad_(False)
        self.enabled = True

    def update(self, model):
        self.updates += 1
        d = self.decay(self.updates)
        msd = (model.module if hasattr(model, "module") else model).state_dict()
        for k, v in self.ema.state_dict().items():
            if v.dtype.is_floating_point:
                v *= d
                v += (1 - d) * msd[k].detach()

    def update_attr(self, model, include=(), exclude=("process_group", "reducer")):
        copy_attr(self.ema, model, include, exclude)


def model_info(model, detailed=False, verbose=True, imgsz=640):
    n_p = sum(x.numel() for x in model.parameters())
    n_l = len(list(model.modules()))
    return n_l, n_p, 0, 0.0


def time_sync():
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    return time.time()


def intersect_dicts(da, db, exclude=()):
    return {k: v for k, v in da.items() if k in db and all(x not in k for x in exclude) and v.shape == db[k].shape}


def one_cycle(y1=0.0, y2=1.0, steps=100):
    return lambda x: max((1 - math.cos(x * math.pi / steps)) / 2, 0) * (y2 - y1) + y1


def autocast(enabled, device="cuda"):
    return torch.amp.autocast(device, enabled=enabled)


# ----------------------------------------------------------------------------------------------------------------------
# ultralytics.utils (logging & misc helpers; behaviour irrelevant to the arithmetic)
# ----------------------------------------------------------------------------------------------------------------------
LOGGER = logging.getLogger("ref_shim")
LOGGER.addHandler(logging.NullHandler())
LOGGER.setLevel(logging.ERROR)


def colorstr(*inp):
    return str(inp[-1]) if inp else ""


def emojis(s=""):
    return s


class TryExcept(contextlib.ContextDecorator):
    def __init__(self, msg="", verbose=True):
        self.msg = msg

    def __enter__(self):
        return self

    def __exit__(self, exc_type, value, tb):
        return True


def threaded(func):
    def wrapper(*a, **k):
        import threading

        t = threading.Thread(target=func, args=a, kwargs=k, daemon=True)
        t.start()
        return t

    return wrapper


def get_default_args(func):
    import inspect

    sig = inspect.signature(func)
    return {k: v.default for k, v in sig.parameters.items() if v.default is not inspect.Parameter.empty}


def TQDM(it=None, *a, **k):
    from tqdm import tqdm

    k.pop("bar_format", None)
    return tqdm(it, *a, disable=True, **k)


def check_version(current="0.0.0", required="0.0.0", name="version", hard=False, verbose=False, msg=""):
    from packaging.version import parse

    cur = parse(str(current).split("+")[0])
    ok = True
    for r in str(required).strip(",").split(","):
        r = r.strip()
        op = "".join(ch for ch in r[:2] if ch in "<>=!")
        ver = parse(r[len(op):] or "0")
        op = op or ">="
        ok &= {"==": cur == ver, "!=": cur != ver, ">=": cur >= ver, "<=": cur <= ver, ">": cur > ver, "<": cur < ver}[op]
    return ok


def increment_path(path, exist_ok=False, sep="", mkdir=False):
    path = Path(path)
    if path.exists() and not exist_ok:
        base, suf = (path.with_suffix(""), path.suffix) if path.is_file() else (path, "")
        for n in range(2, 9999):
            p = f"{base}{sep}{n}{suf}"
            if not Path(p).exists():
                break
        path = Path(p)
    if mkdir:
        path.mkdir(parents=True, exist_ok=True)
    return path


class WorkingDirectory(contextlib.ContextDecorator):
    def __init__(self, new_dir):
        self.dir = new_dir
        self.cwd = Path.cwd().resolve()

    def __enter__(self):
        import os

        os.chdir(self.dir)

    def __exit__(self, *a):
        import os

        os.chdir(self.cwd)


class GitRepo:
    def __init__(self, path=None):
        self.root = None
        self.origin = None
        self.branch = None
        self.commit = None


class _Annotator:
    def __init__(self, im, *a, **k):
        self.im = im

    def box_label(self, *a, **k):
        pass

    def result(self):
        return self.im


def _module(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def install():
    """Register the stand-in modules and put ``REFERENCE_ROOT`` on sys.path.  Idempotent."""
    if "ultralytics" in sys.modules and getattr(sys.modules["ultralytics"], "_y3_shim", False):
        return
    noop = lambda *a, **k: None  # noqa: E731
    u = _module("ultralytics", _y3_shim=True, __version__="8.4.110", __path__=[])
    _module("ultralytics.utils", LOGGER=LOGGER, TQDM=TQDM, colorstr=colorstr, emojis=emojis, TryExcept=TryExcept,
            threaded=threaded, get_default_args=get_default_args, __path__=[])
    _module("ultralytics.utils.checks", check_requirements=noop, check_version=check_version,
            is_ascii=lambda s="": all(ord(c) < 128 for c in str(s)), print_args=noop)
    _module("ultralytics.utils.files", WorkingDirectory=WorkingDirectory, file_date=lambda p=__file__: "1970-1-1",
            file_size=lambda p: 0.0, get_latest_run=lambda search_dir=".": "", increment_path=increment_path)
    _module("ultralytics.utils.git", GitRepo=GitRepo)
    _module("ultralytics.utils.ops", Profile=Profile, clip_boxes=clip_boxes, make_divisible=make_divisible,
            xywh2xyxy=xywh2xyxy, xywhn2xyxy=xywhn2xyxy, xyxy2xywh=xyxy2xywh, xyxy2xywhn=xyxy2xywhn)
    _module("ultralytics.utils.patches", torch_load=lambda *a, **k: torch.load(*a, **{**k, "weights_only": False}))
    _module("ultralytics.utils.torch_utils", ModelEMA=ModelEMA, copy_attr=copy_attr, fuse_conv_and_bn=fuse_conv_and_bn,
            initialize_weights=initialize_weights, model_info=model_info, scale_img=scale_img, time_sync=time_sync,
            intersect_dicts=intersect_dicts, one_cycle=one_cycle, autocast=autocast, TORCH_2_4=True)
    _module("ultralytics.utils.metrics", box_iou=box_iou, bbox_iou=bbox_iou, bbox_ioa=bbox_ioa, smooth_bce=smooth_bce,
            smooth=smooth, plot_mc_curve=noop, plot_pr_curve=noop)
    _module("ultralytics.utils.plotting", Annotator=_Annotator, colors=lambda i, bgr=False: (0, 0, 0),
            save_one_box=noop)
    _module("ultralytics.data", __path__=[])
    _module("ultralytics.data.build", seed_worker=noop)
    _module("ultralytics.data.utils", get_hash=lambda paths: "0", img2label_paths=lambda p: p)
    _module("ultralytics.data.converter", coco80_to_coco91_class=lambda: list(range(1, 92)))
    del u
    if "matplotlib" not in sys.modules:
        try:
            import matplotlib  # noqa: F401
        except ImportError:
            mpl = _module("matplotlib", rc=noop, use=noop, __path__=[])
            mpl.pyplot = _module("matplotlib.pyplot")
    if "seaborn" not in sys.modules:
        try:
            import seaborn  # noqa: F401
        except ImportError:
            _module("seaborn")
    if str(REFERENCE_ROOT) not in sys.path:
        sys.path.insert(0, str(REFERENCE_ROOT))


def reference_available() -> bool:
    return (REFERENCE_ROOT / "models" / "yolo.py").exists()

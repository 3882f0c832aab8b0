"""yolov3_b200 — Blackwell-native (sm_100a) YOLOv3 detection hot path behind the ultralytics/yolov3 Python seams.

Public surface mirrors the reference's (SURVEY.md §8b); every name below resolves lazily to its module (importing the package
costs nothing and never touches the GPU).  All compute runs in the hand-written CUDA library ``libyolov3_b200.so`` through
the C ABI in ``include/yolov3_b200.h``; there is no CPU or PyTorch fallback.

    Model, DetectionModel      models/yolo.py:193 (plain engine front-end / the same object as an nn.Module)
    DetectMultiBackend         models/common.py:435
    non_max_suppression        utils/general.py:630      (nms_batched: the sync-free padded form)
    scale_boxes, clip_boxes    utils/general.py:613-626
    box_iou                    utils/metrics.py:10
    process_batch              val.py:147
    ap_per_class, ConfusionMatrix   utils/metrics.py:22, :124 (ap_per_class_batched: the sync-free padded form)
    ComputeLoss                utils/loss.py:98
    letterbox                  utils/augmentations.py:104 (preprocess.preprocess: + utils/dataloaders.py:308-310 layout step)
    forward_augment, Ensemble, attempt_load   models/yolo.py:239-280, models/experimental.py:74-136
    DDP, scale_loss, convert_sync_batchnorm   utils/torch_utils.py:60-72, train.py:405-406, :270-272
    SGD, ModelEMA              utils/torch_utils.py:207-237 + train.py:411-421 (fused clip + SGD-nesterov + EMA)
    Pipeline                   detect.py:185-200 loop body
"""
import importlib

__version__ = "0.2.0"

_EXPORTS = {
    "Model": "model", "Engine": "model", "DetectionModel": "module", "DetectMultiBackend": "backend", "save_checkpoint": "backend",
    "non_max_suppression": "nms", "nms_batched": "nms", "scale_boxes": "boxes", "clip_boxes": "boxes", "box_iou": "loss",
    "ComputeLoss": "loss", "process_batch": "val", "process_batch_batched": "val", "letterbox": "preprocess",
    "forward_augment": "tta", "Ensemble": "tta", "attempt_load": "tta", "DDP": "parallel",
    "scale_loss": "parallel", "convert_sync_batchnorm": "parallel", "SGD": "optim", "ModelEMA": "optim", "Pipeline": "pipeline",
    "ap_per_class": "metrics", "ap_per_class_batched": "metrics", "ConfusionMatrix": "metrics",
}
__all__ = sorted(_EXPORTS)


def __getattr__(name):
    mod = _EXPORTS.get(name)
    if mod is None:
        raise AttributeError(f"module 'yolov3_b200' has no attribute {name!r}")
    return getattr(importlib.import_module(f"{__name__}.{mod}"), name)


def __dir__():
    return sorted(list(globals()) + list(_EXPORTS))

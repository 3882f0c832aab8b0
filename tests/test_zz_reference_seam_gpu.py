"""The seam with the REFERENCE's own scripts, checked against what they computed (tests/golden/seam_cases.npz, written by
tests/golden/make_golden.py from the unmodified reference): detect.py's loop with our ``DetectMultiBackend``,
``non_max_suppression`` and ``scale_boxes`` on the reference's sample images, the val.py loop body, and train.py's optimizer
groups / EMA on the nn.Module facade."""
from pathlib import Path

import numpy as np
import pytest
import torch

import yolo_oracle as O

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
CFG = ROOT / "yolov3_b200" / "cfg"
GOLDEN = ROOT / "tests" / "golden" / "seam_cases.npz"


def rel_l2(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


def test_detect_loop_on_our_backend_matches_reference(tmp_path):
    """BASELINE config 1 plumbing with the backend swapped in: detect.py's calls (detect.py:166-223) on our
    DetectMultiBackend / non_max_suppression / scale_boxes over the reference's data/images (letterboxed by its LoadImages)
    find detections; image by image, our forward vs the reference model's (rel-L2 <= 2e-2) and — on the reference's own
    predictions — our NMS + scale_boxes vs the reference's (bit-exact)."""
    from yolov3_b200 import backend, boxes, nms
    from yolov3_b200.model import Model

    g = np.load(GOLDEN)
    cfg = CFG / "yolov3-tiny.yaml"
    m = Model(cfg)
    m.load_state_dict(O.confident_params(cfg))
    ckpt = tmp_path / "tiny_b200.pt"
    backend.save_checkpoint(m, ckpt)
    model = backend.DetectMultiBackend(str(ckpt), device=torch.device("cuda"), dnn=False, data=None, fp16=False)
    assert model.pt and model.stride == 32 and len(model.names) == 80
    n_img = len({k.split("/")[1] for k in g.files if k.startswith("detect/")})
    assert n_img == 2
    for i in range(n_img):
        im, shape0 = g[f"detect/{i}/im"], tuple(int(v) for v in g[f"detect/{i}/im0_shape"])
        model.warmup(imgsz=(1, 3, *im.shape[1:]))
        x = model.from_numpy(im).float()[None] / 255
        pred = model(x, augment=False, visualize=False)
        det = nms.non_max_suppression(pred, 0.25, 0.45, None, False, max_det=50)[0]
        assert len(det) >= 1, i
        det[:, :4] = boxes.scale_boxes(x.shape[2:], det[:, :4], shape0).round()
        assert bool((det[:, [0, 2]] <= shape0[1]).all() and (det[:, [1, 3]] <= shape0[0]).all() and (det[:, :4] >= 0).all())
        # ---- parity of the swapped pieces on the same image
        z_ref = torch.from_numpy(g[f"detect/{i}/z"])
        assert rel_l2(pred[0], z_ref) <= 2e-2, i
        det_ref = g[f"detect/{i}/det"]
        det = nms.non_max_suppression(z_ref.cuda(), 0.25, 0.45, max_det=50)[0]
        # real-image predictions with saturating sigmoids contain bit-equal confidences (birthday collisions among the
        # candidates): the reference orders such ties by an unstable argsort, we by candidate index — compare row SETS
        # (rows sorted lexicographically), which is what "identical detections" means when the order is undefined
        a, b = det_ref, det.cpu().numpy()
        assert a.shape == b.shape, (i, a.shape, b.shape)
        ka = np.lexsort(a.T[::-1])
        kb = np.lexsort(b.T[::-1])
        assert np.array_equal(a[ka], b[kb]), (i, np.abs(a[ka] - b[kb]).max())
        det = torch.from_numpy(det_ref).cuda()  # continue with identical rows in identical order
        sb = boxes.scale_boxes(x.shape[2:], det[:, :4].clone(), shape0)
        assert np.array_equal(sb.cpu().numpy(), g[f"detect/{i}/scaled"])


def test_val_loop_body_pieces_match_reference():
    """val.py:355-390 with our pieces: NMS (multi-label, conf 0.001, iou 0.6), scale_boxes to native space and
    process_batch give exactly the reference's detections and ``correct`` matrix."""
    from ref_shim import xywh2xyxy  # the shim's restatement of the third-party function

    from yolov3_b200 import boxes, nms
    from yolov3_b200.val import process_batch

    g = np.load(GOLDEN)
    pred = O.synth_predictions(2, n_rows=3000, nc=80, seed=5)
    targets = O.synth_targets(2, seed=4)
    h = w = 640
    shape0, ratio_pad = (480, 600), ((1.0667, 1.0667), (0.0, 64.0))
    targets_px = targets.clone()
    targets_px[:, 2:] *= torch.tensor((w, h, w, h))
    iouv = torch.linspace(0.5, 0.95, 10)
    our_out = nms.non_max_suppression(pred.cuda(), 0.001, 0.6, multi_label=True, max_det=300)
    for si in range(2):
        labels = targets_px[targets_px[:, 0] == si, 1:]
        predn = our_out[si].clone()
        assert np.array_equal(predn.cpu().numpy(), g[f"val/{si}/out"])
        boxes.scale_boxes((h, w), predn[:, :4], shape0, ratio_pad)
        tb = xywh2xyxy(labels[:, 1:5]).cuda()
        boxes.scale_boxes((h, w), tb, shape0, ratio_pad)
        labelsn = torch.cat((labels[:, 0:1].cuda(), tb), 1)
        assert np.array_equal(labelsn.cpu().numpy(), g[f"val/{si}/labelsn"])
        correct = process_batch(predn, labelsn, iouv.cuda())
        assert np.array_equal(predn.cpu().numpy(), g[f"val/{si}/predn"])
        assert np.array_equal(correct.cpu().numpy(), g[f"val/{si}/correct"]), si


def reference_sgd(model, name):
    """torch.optim.SGD with the parameter groups the reference's ``smart_optimizer(model, "SGD", 0.01, 0.937, 5e-4)``
    (utils/torch_utils.py:207-237) forms, taken by name from the fixture."""
    g = np.load(GOLDEN)
    params = dict(model.named_parameters())
    groups = []
    for gi in range(3):
        lr, momentum, dampening, decay, nesterov = (float(v) for v in g[f"optim/{name}/{gi}/hyp"])
        groups.append(dict(params=[params[n] for n in g[f"optim/{name}/{gi}/names"]], lr=lr, momentum=momentum,
                           dampening=dampening, weight_decay=decay, nesterov=bool(nesterov)))
    return torch.optim.SGD(groups)


def _train_two_steps(model, opt_step, zero_grad, x, targets, loss_fn):
    losses = []
    for _ in range(2):
        pred = model(x)
        loss, _ = loss_fn(pred, targets)
        loss.backward()
        opt_step()
        zero_grad()
        losses.append(float(loss.detach()))
    return losses


def test_facade_with_reference_optimizer_and_ema():
    """train.py's objects on the facade: the three parameter groups of ``smart_optimizer`` (utils/torch_utils.py:207-237),
    ``ModelEMA`` (train.py:252) deep-copies and updates, ``clip_grad_norm_`` + ``optimizer.step()`` train the masters —
    and two steps land where our fused step (optim.SGD + ModelEMA) lands on an identically initialised model."""
    from ref_shim import ModelEMA as RefEMA  # the shim's restatement of the third-party class

    from yolov3_b200.loss import ComputeLoss
    from yolov3_b200.module import DetectionModel
    from yolov3_b200.optim import SGD, ModelEMA
    from yolov3_b200.train import TrainEngine

    TrainEngine.deterministic = True
    try:
        cfg = CFG / "yolov3.yaml"
        params = O.init_params(cfg, seed=0)
        x = torch.rand(2, 3, 64, 64, generator=torch.Generator().manual_seed(3)).cuda()
        targets = O.synth_targets(2, seed=2).cuda()
        hyp = O.scaled_hyp()
        # ---- A: facade + reference optimizer + reference-style EMA
        ma = DetectionModel(cfg)
        ma.load_state_dict(params, strict=False)
        ma.hyp = hyp
        names = {n for n, _ in ma.named_parameters()}
        assert "model.4.0.cv1.conv.weight" in names and "model.28.m.2.bias" in names and len(names) == 222
        opt = reference_sgd(ma, "yolov3")
        assert [len(g["params"]) for g in opt.param_groups] == [75, 75, 72]  # biases (72 BN + 3 head), decay weights, BN weights
        ema = RefEMA(ma)
        ma.train()
        loss_fn = ComputeLoss(ma)

        def step_a():
            torch.nn.utils.clip_grad_norm_(ma.parameters(), max_norm=10.0)
            opt.step()
            ema.update(ma)

        la = _train_two_steps(ma, step_a, opt.zero_grad, x, targets, loss_fn)
        # ---- B: plain Model + fused optimizer
        mb = DetectionModel(cfg)
        mb.load_state_dict(params, strict=False)
        mb.hyp = hyp
        mb.train()
        ema_b = ModelEMA(mb.core)
        opt_b = SGD(mb.core, lr=0.01, momentum=0.937, weight_decay=5e-4, nesterov=True, max_norm=10.0, ema=ema_b)
        lb = _train_two_steps(mb, opt_b.step, opt_b.zero_grad, x, targets, ComputeLoss(mb))
        assert la == lb, (la, lb)  # deterministic engines, identical updates after step 1 -> identical loss at step 2
        sa, sb = ma.state_dict(), mb.state_dict()
        for k in sa:
            if "num_batches_tracked" in k:
                continue
            assert torch.allclose(sa[k].float(), sb[k].float(), rtol=1e-5, atol=1e-7), k
        ea, eb = ema.ema.state_dict(), ema_b.state_dict()
        for k in eb:
            assert torch.allclose(ea[k].float().cpu(), eb[k], rtol=1e-5, atol=1e-7), k
        # eval-mode inference picks the trained weights up (in-place updates are detected through the store's version)
        ma.eval()
        mb.eval()
        za, zb = ma(x)[0], mb(x)[0]
        assert torch.equal(za, zb) and bool(torch.isfinite(za).all())
        # half(): fp16 outputs, masters rounded to fp16-representable values (train.py:317)
        zh = ma.half()(x.half())[0]
        assert zh.dtype == torch.float16
        w = ma.state_dict()["model.5.conv.weight"]
        assert torch.equal(w, w.half().float())
    finally:
        TrainEngine.deterministic = False

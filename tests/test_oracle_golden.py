"""The CPU oracle (oracle/yolo_oracle.py) against the golden fixtures produced by the reference itself
(tests/golden/make_golden.py).  Runs everywhere (no GPU, no /root/reference)."""
import ast
from pathlib import Path

import numpy as np
import pytest
import torch

import yolo_oracle as O

G = Path(__file__).parent / "golden"
CFG = Path(__file__).resolve().parents[1] / "yolov3_b200" / "cfg"


@pytest.mark.parametrize("name", ["yolov3-tiny", "yolov3", "yolov3-spp"])
def test_forward_matches_reference(name):
    g = np.load(G / f"forward_{name}.npz")
    params = O.init_params(CFG / f"{name}.yaml", seed=int(g["param_seed"]))
    om = O.OracleModel(CFG / f"{name}.yaml", params=params, fused=True)
    assert om.save == list(g["save"]) and np.array_equal(om.stride.numpy(), g["stride"])
    ci = 0
    while f"z{ci}" in g:
        bs, c, h, w = g[f"x{ci}_shape"]
        x = torch.rand(int(bs), int(c), int(h), int(w), generator=torch.Generator().manual_seed(int(g[f"x{ci}_seed"])))
        taps = {int(k.split("_")[1]): None for k in g.files if k.startswith(f"tap{ci}_")}
        with torch.no_grad():
            z, raw = om(x, taps)
        assert np.allclose(z.numpy(), g[f"z{ci}"], atol=2e-4, rtol=2e-4)
        for li, r in enumerate(raw):
            assert np.allclose(r.numpy(), g[f"raw{ci}_{li}"], atol=2e-4, rtol=2e-4)
        for i, t in taps.items():
            ref = g[f"tap{ci}_{i}"]
            flat = t.flatten()
            idx = torch.linspace(0, flat.numel() - 1, 64).long()
            got = np.concatenate([[t.mean().item(), t.std().item(), t.abs().max().item()], flat[idx].numpy()])
            assert np.allclose(got, ref, atol=2e-4, rtol=2e-4), (name, ci, i)
        ci += 1
    assert ci >= 1


def _nms_cases():
    g = np.load(G / "nms_cases.npz")
    return sorted({k.split("/")[0] for k in g.files if "/" in k})


@pytest.mark.parametrize("case", _nms_cases())
def test_nms_bit_exact(case):
    g = np.load(G / "nms_cases.npz")
    kw = ast.literal_eval(str(g[f"{case}/kw"]))
    pred = g[str(g[f"{case}/pred_key"])]
    outs, srcs = O.non_max_suppression(torch.from_numpy(pred), **kw)
    for xi, (o, s) in enumerate(zip(outs, srcs)):
        assert np.array_equal(o, g[f"{case}/out{xi}"])
        assert np.array_equal(s, g[f"{case}/src{xi}"])


@pytest.mark.parametrize("case", range(4))
def test_loss_matches_reference(case):
    import sys
    sys.path.insert(0, str(G))
    from make_golden import loss_inputs

    g = np.load(G / "loss_cases.npz")
    hyp = ast.literal_eval(str(g["hyp"]))
    anchors = torch.from_numpy(g["anchors"])
    p, t = loss_inputs(case)
    assert np.array_equal(t.numpy(), g[f"c{case}/targets"])
    p = [x.requires_grad_(True) for x in p]
    loss, items = O.compute_loss(p, t, anchors, hyp)
    loss.backward()
    assert np.allclose(loss.detach().numpy(), g[f"c{case}/loss"], rtol=1e-5)
    assert np.allclose(items.numpy(), g[f"c{case}/items"], rtol=1e-5, atol=1e-7)
    for i, x in enumerate(p):
        assert np.allclose(x.grad.numpy(), g[f"c{case}/grad{i}"], rtol=1e-4, atol=1e-7)
    bt = O.build_targets([tuple(x.shape) for x in p], t, anchors, hyp["anchor_t"])
    for i in range(3):
        got = torch.cat((torch.stack([bt[i][k].float() for k in ("b", "a", "gj", "gi")], 1), bt[i]["tbox"], bt[i]["anch"],
                         bt[i]["tcls"][:, None].float()), 1).numpy()
        assert np.allclose(got, g[f"c{case}/bt{i}"], atol=1e-6)


def test_iou():
    g = np.load(G / "iou_cases.npz")
    assert np.array_equal(O.box_iou(g["a"], g["b"]).numpy(), g["iou"])
    assert np.allclose(O.ciou_xywh(torch.from_numpy(g["p1"]), torch.from_numpy(g["p2"])).numpy(), g["ciou"], atol=1e-6)


def test_scale_boxes_bit_exact():
    """oracle scale_boxes == reference utils/general.py:613-626 on the committed fixtures (4 letterbox geometries)."""
    g = np.load(G / "scale_boxes_cases.npz")
    for ci in range(sum(k.startswith("geom") for k in g.files)):
        s1, s0, rp = ast.literal_eval(str(g[f"geom{ci}"]))
        out = O.scale_boxes(s1, g[f"in{ci}"][:, :4], s0, rp)
        assert np.array_equal(out, g[f"out{ci}"][:, :4])


def test_oracle_greedy_nms_equals_torchvision():
    """The numpy greedy pass of the oracle and torchvision.ops.nms (what the reference calls, general.py:733) keep the same
    boxes in the same order on the config-5 workload."""
    pred = O.synth_predictions(2, n_rows=25200, nc=80, seed=3)
    for conf, iou, ml in ((0.25, 0.45, False), (0.05, 0.45, True)):
        a, sa = O.non_max_suppression(pred, conf, iou, multi_label=ml)
        b, sb = O.non_max_suppression(pred, conf, iou, multi_label=ml, use_torchvision=True)
        for x, y, sx, sy in zip(a, b, sa, sb):
            assert np.array_equal(x, y) and np.array_equal(sx, sy)


def test_oracle_nms_properties():
    """Size-independent properties of the checker itself: rows sorted by confidence, every kept score above the
    threshold, kept boxes of one class never overlap above the IoU threshold, idempotence (NMS of its own output keeps
    everything), and invariance of the kept set under a permutation of the prediction rows."""
    pred = O.synth_predictions(1, n_rows=4000, nc=80, seed=9)
    conf, iou = 0.1, 0.45
    (out,), (src,) = O.non_max_suppression(pred, conf, iou, max_det=1000)
    assert out.shape[0] > 10 and np.all(out[:-1, 4] >= out[1:, 4]) and np.all(out[:, 4] > conf)
    for c in np.unique(out[:, 5]):
        b = out[out[:, 5] == c][:, :4]
        if len(b) > 1:
            m = O.box_iou(torch.from_numpy(b), torch.from_numpy(b)).numpy()
            np.fill_diagonal(m, 0.0)
            assert m.max() <= iou + 1e-6
    again = torch.zeros(1, out.shape[0], 85)
    again[0, :, 0:2] = torch.from_numpy((out[:, 0:2] + out[:, 2:4]) / 2)
    again[0, :, 2:4] = torch.from_numpy(out[:, 2:4] - out[:, 0:2])
    again[0, :, 4] = 1.0
    again[0, torch.arange(out.shape[0]), 5 + torch.from_numpy(out[:, 5]).long()] = torch.from_numpy(out[:, 4])
    (out2,), _ = O.non_max_suppression(again, conf, iou, max_det=1000)
    assert out2.shape[0] == out.shape[0]
    perm = torch.randperm(pred.shape[1], generator=torch.Generator().manual_seed(1))
    (out3,), (src3,) = O.non_max_suppression(pred[:, perm], conf, iou, max_det=1000)
    assert np.array_equal(out3, out) and np.array_equal(perm.numpy()[src3[:, 0]], src[:, 0])


def test_process_batch_oracle_vs_reference_golden():
    """oracle.process_batch (restatement of val.py:147-188) against the matrices the reference's own val.process_batch produced."""
    g = np.load(G / "val_cases.npz")
    iouv = torch.from_numpy(g["iouv"])
    for case in sorted({k.split("/")[0] for k in g.files if "/" in k}):
        det, lab = torch.from_numpy(g[f"{case}/det"]), torch.from_numpy(g[f"{case}/lab"])
        if lab.shape[0] == 0:
            continue
        assert np.array_equal(O.process_batch(det, lab, iouv).numpy(), g[f"{case}/correct"]), case
        d2, l2 = O.synth_val_case(det.shape[0], lab.shape[0], 6, seed=0)  # the generator is part of the fixture contract
    d0, l0 = O.synth_val_case(120, 25, 6, 0, 12.0)
    assert np.array_equal(d0.numpy(), g["typical/det"]) and np.array_equal(l0.numpy(), g["typical/lab"])


def test_letterbox_oracle_vs_cv2_and_reference():
    """oracle.resize_linear_u8 / letterbox (restating OpenCV's 8-bit INTER_LINEAR and utils/augmentations.py:104-134) against
    cv2 itself (third-party, installed: opencv-python 4.13) and the reference's own letterbox() (seam_cases.npz: digest of
    its image, ratio and padding on seeded random images)."""
    import hashlib

    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(0)
    for (h, w, nh, nw) in [(480, 640, 480, 640), (1080, 810, 640, 480), (720, 1280, 360, 640), (375, 500, 480, 640), (100, 133, 640, 851),
                           (501, 333, 417, 277), (64, 64, 200, 31), (33, 77, 32, 75)]:
        im = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert np.array_equal(O.resize_linear_u8(im, nw, nh), cv2.resize(im, (nw, nh), interpolation=cv2.INTER_LINEAR)), (h, w, nh, nw)
    g = np.load(G / "seam_cases.npz")
    rng = np.random.default_rng(1)
    for i, (h, w) in enumerate(g["letterbox/shapes"]):
        im = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        for k, kw in enumerate(ast.literal_eval(str(g["letterbox/kw"]))):
            b = O.letterbox(im.copy(), **kw)
            assert b[0].shape == tuple(g[f"letterbox/{i}_{k}/shape"]), (i, k)
            assert hashlib.sha256(np.ascontiguousarray(b[0]).tobytes()).hexdigest() == str(g[f"letterbox/{i}_{k}/sha256"]), (i, k)
            assert tuple(b[1]) == tuple(g[f"letterbox/{i}_{k}/ratio"]) and tuple(b[2]) == tuple(g[f"letterbox/{i}_{k}/pad"]), (i, k)

"""Validation metrics on the device (y3_ap_per_class, y3_confusion_update) against the goldens recorded from the reference's
own ap_per_class / ConfusionMatrix (tests/golden/make_metrics_golden.py) and, at COCO-val size, against the CPU restatement
in tests/metrics_oracle.py.  AP bit-identical, p / r / f1 within 1e-12, counts and matrices exact."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent))
import metrics_oracle as MO  # noqa: E402
import yolo_oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu
G = Path(__file__).parent / "golden"
TOL = 1e-12


def _cases(prefix):
    g = np.load(G / "metrics_cases.npz")
    return sorted({k.split("/")[1] for k in g.files if k.startswith(prefix + "/")})


def _flat_batched(tp, conf, pred_cls, target_cls, nc):
    """The same rows as one image of the padded layout (no counts) through ap_per_class_batched."""
    from yolov3_b200.metrics import ap_per_class_batched

    n = len(conf)
    det = torch.zeros(1, n, 6)
    det[0, :, 4], det[0, :, 5] = torch.from_numpy(conf), torch.from_numpy(pred_cls)
    labels = torch.zeros(len(target_cls), 6)
    labels[:, 1] = torch.from_numpy(target_cls)
    return ap_per_class_batched(det.cuda(), None, torch.from_numpy(tp).reshape(1, n, -1).cuda(), labels.cuda(), nc)


@pytest.mark.parametrize("case", _cases("ap"))
def test_ap_per_class_golden(case):
    from yolov3_b200.metrics import ap_per_class

    g = np.load(G / "metrics_cases.npz")
    k = f"ap/{case}/"
    tp, conf, pc, tc = g[k + "tp"], g[k + "conf"], g[k + "pred_cls"], g[k + "target_cls"]
    out = ap_per_class(tp, conf, pc, tc)
    names = ("out_tp", "out_fp", "p", "r", "f1", "ap", "cls")
    for got, key in zip(out, names):
        ref = g[k + key]
        assert got.dtype == ref.dtype and got.shape == ref.shape, (key, got.dtype, ref.dtype, got.shape, ref.shape)
        if key in ("p", "r", "f1"):
            assert np.allclose(got, ref, rtol=0, atol=TOL), key
        else:
            assert np.array_equal(got, ref), key
    # the padded form on the same rows: the same numbers, and the F1 index the reference chose
    b = _flat_batched(tp, conf, pc, tc, int(tc.max()) + 1)
    cls = g[k + "cls"]
    assert int(b.f1_index.item()) == int(g[k + "i"])
    assert np.array_equal(b.ap.cpu().numpy()[cls], out[5]) and np.array_equal(b.p.cpu().numpy()[cls], out[2])
    assert np.array_equal(np.flatnonzero(b.present.cpu().numpy()), cls)
    assert np.array_equal(b.nt.cpu().numpy()[cls], np.bincount(tc.astype(int))[cls])
    nc = int(tc.max()) + 1  # predictions of a class beyond every label's (pred_no_label) are counted, then ignored
    assert b.status.cpu().tolist() == [int((pc >= nc).sum()), 0, 0]


def _cm_golden_case(case):
    g = np.load(G / "metrics_cases.npz")
    k = f"cm/{case}/"
    return int(g[k + "nc"]), g[k + "det"], g[k + "counts"], g[k + "labels"], g[k + "matrix"]


@pytest.mark.parametrize("case", _cases("cm"))
def test_confusion_matrix_golden_batched_and_per_image(case):
    from yolov3_b200.metrics import ConfusionMatrix

    nc, det, counts, labels, ref = _cm_golden_case(case)
    cm = ConfusionMatrix(nc)
    cm.process_batch_batched(torch.from_numpy(det).cuda(), torch.from_numpy(counts).cuda(), torch.from_numpy(labels).cuda())
    assert cm.matrix.dtype == np.float64 and np.array_equal(cm.matrix, ref)
    per = ConfusionMatrix(nc)
    for i in range(len(counts)):  # val.py:390,406
        lab = torch.from_numpy(labels[labels[:, 0] == i, 1:]).cuda()
        if counts[i] < 0:
            per.process_batch(detections=None, labels=lab[:, 0])
        else:
            per.process_batch(torch.from_numpy(det[i, : counts[i]]).cuda(), lab)
    assert np.array_equal(per.matrix, ref)
    tp, fp = per.tp_fp()
    assert np.array_equal(tp, ref.diagonal()[:-1]) and np.array_equal(fp, (ref.sum(1) - ref.diagonal())[:-1])
    assert per.invalid == (0, 0)


def _coco_sized(seed=0, nimg=5000, max_det=300, nc=80, niou=10):
    """nms_batched / process_batch_batched-shaped stats: [nimg, max_det, 6] + random counts + correct; padded rows hold
    garbage (high confidence, true positive) that must be ignored."""
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, max_det + 1, nimg).astype(np.int32)
    counts[:3] = (0, max_det, 1)
    nvalid = int(counts.sum())
    tp, conf, pc, tc = MO.synth_stats(nvalid, nc, n_targets=7 * nimg, niou=niou, seed=seed + 1)
    valid = (np.arange(max_det)[None, :] < counts[:, None]).reshape(-1)
    det = np.zeros((nimg * max_det, 6), np.float32)
    det[:, 4], det[:, 5] = 0.999, rng.integers(0, nc, nimg * max_det)
    det[valid, 4], det[valid, 5] = conf, pc
    correct = np.ones((nimg * max_det, niou), bool)
    correct[valid] = tp
    labels = np.zeros((len(tc), 6), np.float32)
    labels[:, 0], labels[:, 1] = rng.integers(0, 32, len(tc)), tc
    return det.reshape(nimg, max_det, 6), counts, correct.reshape(nimg, max_det, niou), labels, (tp, conf, pc, tc)


def _assert_matches_oracle(res, o):
    """res: APResult (host copies), o: metrics_oracle.ap_per_class dict.  Near-tied smoothed F1 maxima (within 1e-12) may
    pick either index; the comparison is then made at the index the device chose."""
    i = int(res["f1_index"][0])
    if i != o["i"]:
        assert abs(o["f1_smooth"][i] - o["f1_smooth"][o["i"]]) <= TOL, (i, o["i"])
        present = o["present"]
        p, r = o["pcurve"][:, i] * present, o["rcurve"][:, i] * present
        f1 = 2 * p * r / (p + r + 1e-16)
        tpo = np.round(r * o["nt"])
        o = dict(o, p=p, r=r, f1=f1, tp=tpo, fp=np.round(tpo / (p + 1e-16) - tpo))
    assert np.array_equal(res["ap"], o["ap"])
    for key in ("p", "r", "f1"):
        assert np.allclose(res[key], o[key], rtol=0, atol=TOL), key
    assert np.array_equal(res["tp"], o["tp"]) and np.array_equal(res["fp"], o["fp"])
    assert np.array_equal(res["nt"], o["nt"]) and np.array_equal(res["present"], o["present"])


def _host(res):
    return {k: v.cpu().numpy() for k, v in res._asdict().items()}


def test_ap_per_class_coco_sized_matches_oracle_batched_equals_dropin_deterministic_no_sync():
    from yolov3_b200.metrics import ap_per_class, ap_per_class_batched

    det, counts, correct, labels, (tp, conf, pc, tc) = _coco_sized()
    d_det, d_counts = torch.from_numpy(det).cuda(), torch.from_numpy(counts).cuda()
    d_correct, d_labels = torch.from_numpy(correct).cuda(), torch.from_numpy(labels).cuda()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        a = ap_per_class_batched(d_det, d_counts, d_correct, d_labels, 80)
        b = ap_per_class_batched(d_det, d_counts, d_correct, d_labels, 80)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    ha, hb = _host(a), _host(b)
    for k in ha:
        assert np.array_equal(ha[k], hb[k]), k  # deterministic
    assert ha["status"].tolist() == [0, 0, 0]
    _assert_matches_oracle(ha, MO.ap_per_class(tp, conf, pc, tc, nc=80))
    # the drop-in on the concatenated valid rows gives bit-identical numbers
    out = ap_per_class(tp, conf, pc, tc)
    cls = np.flatnonzero(ha["present"])
    for got, key in zip(out, ("tp", "fp", "p", "r", "f1", "ap")):
        assert np.array_equal(got, ha[key][cls]), key
    assert np.array_equal(out[6], cls)


def test_ap_per_class_confidence_ties_follow_row_order():
    from yolov3_b200.metrics import ap_per_class

    tp, conf, pc, tc = MO.synth_stats(20000, 12, 3000, seed=7, ties=True)
    assert len(np.unique(conf)) < 50
    res = ap_per_class(tp, conf, pc, tc)
    o = MO.ap_per_class(tp, conf, pc, tc)["ref"]
    assert np.array_equal(res[5], o[5])  # AP depends on the order inside a tie: the stable row order
    for k in (2, 3, 4):
        assert np.allclose(res[k], o[k], rtol=0, atol=TOL)
    # reversing the rows of a tie group changes the stable order, and the result follows the oracle on that order too
    rev = np.arange(len(conf))[::-1].copy()
    res_r = ap_per_class(tp[rev], conf[rev], pc[rev], tc)
    assert np.array_equal(res_r[5], MO.ap_per_class(tp[rev], conf[rev], pc[rev], tc)["ref"][5])


def test_ap_per_class_edges():
    from yolov3_b200.metrics import ap_per_class, ap_per_class_batched

    # no predictions at all: every present class has zero rows
    out = ap_per_class(np.zeros((0, 10), bool), np.zeros(0, np.float32), np.zeros(0, np.float32), np.array([2.0, 2.0, 5.0], np.float32))
    assert np.array_equal(out[6], [2, 5]) and not out[5].any() and out[5].shape == (2, 10)
    with pytest.raises(NotImplementedError):
        ap_per_class(np.zeros((1, 10), bool), np.ones(1, np.float32), np.zeros(1, np.float32), np.zeros(1, np.float32), plot=True)
    # out-of-range prediction classes are counted and ignored; labels with such classes are counted
    det = torch.zeros(1, 4, 6)
    det[0, :, 4] = torch.tensor([0.9, 0.8, 0.7, 0.6])
    det[0, :, 5] = torch.tensor([0.0, 85.0, -1.0, 0.0])
    labels = torch.tensor([[0, 0.0, 0, 0, 1, 1], [0, 90.0, 0, 0, 1, 1]])
    correct = torch.zeros(1, 4, 10, dtype=torch.bool)
    correct[0, 0] = True
    r = ap_per_class_batched(det.cuda(), None, correct.cuda(), labels.cuda(), 3)
    assert r.status.cpu().tolist() == [2, 1, 0]
    assert r.present.cpu().tolist() == [True, False, False] and r.nt.cpu().tolist() == [1, 0, 0]
    assert float(r.ap[0, 0]) == MO.ap_per_class(np.array([[1] * 10, [0] * 10], bool), np.array([0.9, 0.6], np.float32),
                                                np.zeros(2, np.float32), np.zeros(1, np.float32))["ap"][0, 0]


def _cm_images(seed, nimg=5000, max_det=300, nc=80):
    """Padded NMS-like batch: labels (image, cls, xyxy) ~7 per image, detections mostly jittered copies of them."""
    rng = np.random.default_rng(seed)
    nl = rng.poisson(7.0, nimg).clip(0, 40)
    img = np.repeat(np.arange(nimg), nl)
    xy = rng.random((len(img), 2)) * 500
    wh = rng.random((len(img), 2)) * 120 + 10
    labels = np.concatenate((img[:, None], rng.integers(0, nc, (len(img), 1)), xy, xy + wh), 1).astype(np.float32)
    counts = rng.integers(0, max_det + 1, nimg).astype(np.int32)
    counts[:4] = (0, 0, max_det, 3)
    det = np.zeros((nimg, max_det, 6), np.float32)
    starts = np.concatenate(([0], np.cumsum(nl)))
    for i in range(nimg):
        n, lab = counts[i], labels[starts[i]:starts[i + 1]]
        src = rng.integers(0, max(len(lab), 1), n)
        box = lab[src, 2:] + rng.normal(0, 6, (n, 4)) if len(lab) else rng.random((n, 4)) * 500
        rnd = rng.random(n) < 0.3
        xy0 = rng.random((int(rnd.sum()), 2)) * 500
        box[rnd] = np.concatenate((xy0, xy0 + 40), 1)
        cls = lab[src, 1] if len(lab) else rng.integers(0, nc, n)
        wrong = rng.random(n) < 0.2
        cls = np.where(wrong, rng.integers(0, nc, n), cls)
        det[i, :n] = np.concatenate((box, np.sort(rng.random(n))[::-1, None], cls[:, None]), 1)
    return det, counts, labels


def test_confusion_matrix_coco_sized_batched_equals_per_image_and_oracle_no_sync():
    from yolov3_b200.metrics import ConfusionMatrix

    det, counts, labels = _cm_images(3)
    nimg, bs = len(counts), 32
    cm = ConfusionMatrix(80)
    batches = []
    for b0 in range(0, nimg, bs):  # labels collated per batch, image index restarting at 0 (collate_fn)
        sel = (labels[:, 0] >= b0) & (labels[:, 0] < b0 + bs)
        lab = labels[sel].copy()
        lab[:, 0] -= b0
        batches.append((torch.from_numpy(det[b0:b0 + bs]).cuda(), torch.from_numpy(counts[b0:b0 + bs]).cuda(),
                        torch.from_numpy(lab).cuda()))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for d, c, lab in batches:
            cm.process_batch_batched(d, c, lab)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    got = cm.matrix
    per = ConfusionMatrix(80)
    ora = np.zeros((81, 81), np.int64)
    for i in range(nimg):
        lab = labels[labels[:, 0] == i, 1:]
        if len(lab) == 0:
            continue  # val.py calls it only for images with labels
        if counts[i] == 0:
            per.process_batch(None, torch.from_numpy(lab[:, 0]).cuda())
            MO.confusion_update(ora, None, lab[:, 0], 80)
        else:
            per.process_batch(torch.from_numpy(det[i, : counts[i]]).cuda(), torch.from_numpy(lab).cuda())
            MO.confusion_update(ora, det[i, : counts[i]], lab, 80)
    assert np.array_equal(got, per.matrix)
    assert np.array_equal(got, ora)
    assert got.sum() > 10000 and cm.invalid == (0, 0)


def test_confusion_matrix_out_of_range_classes_are_counted_not_written():
    from yolov3_b200.metrics import ConfusionMatrix

    det = torch.tensor([[[0, 0, 10, 10, 0.9, 2.0], [20, 20, 30, 30, 0.9, 7.0], [40, 40, 50, 50, 0.9, 1.0]]])
    labels = torch.tensor([[0, 1.0, 0, 0, 10, 10], [0, -4.0, 20, 20, 30, 30], [0, 1.0, 100, 100, 110, 110]])
    cm = ConfusionMatrix(3)
    cm.process_batch_batched(det.cuda(), None, labels.cuda())
    m = np.zeros((4, 4))
    m[2, 1] = 1  # label 0 (class 1) matched by detection 0 (class 2)
    m[3, 1] = 1  # label 2 (class 1) unmatched
    m[1, 3] = 1  # detection 2 (class 1) unmatched; the image has matches
    assert np.array_equal(cm.matrix, m)
    assert cm.invalid == (1, 0)  # label 1 (class -4) matched detection 1 (class 7): one skipped count
    mo = np.zeros((4, 4), np.int64)
    assert MO.confusion_update(mo, det[0].numpy(), labels[:, 1:].numpy(), 3) == 1 and np.array_equal(mo, m)


def test_val_seam_pipeline_reproduces_reference_summary():
    """val.py's loop on the seam's val images, device-only: nms_batched -> scale_boxes -> process_batch_batched ->
    ap_per_class_batched, and the summary of val.py:424-429 from the device results."""
    from ref_shim import xywh2xyxy  # the shim's restatement of the third-party function

    from yolov3_b200 import boxes, nms
    from yolov3_b200.metrics import ap_per_class_batched
    from yolov3_b200.val import process_batch_batched

    g = np.load(G / "metrics_cases.npz")
    pred = O.synth_predictions(2, n_rows=3000, nc=80, seed=5)
    targets = O.synth_targets(2, seed=4)
    h = w = 640
    shape0, ratio_pad = (480, 600), ((1.0667, 1.0667), (0.0, 64.0))
    targets[:, 2:] *= torch.tensor((w, h, w, h))
    iouv = torch.linspace(0.5, 0.95, 10).cuda()
    det, counts, _, _ = nms.nms_batched(pred.cuda(), 0.001, 0.6, multi_label=True, max_det=300)
    predn = det.clone()
    for si in range(2):
        boxes.scale_boxes((h, w), predn[si, : int(counts[si]), :4], shape0, ratio_pad)
    tb = xywh2xyxy(targets[:, 2:6]).cuda()
    boxes.scale_boxes((h, w), tb, shape0, ratio_pad)
    labels = torch.cat((targets[:, :2].cuda(), tb), 1)
    correct = process_batch_batched(predn, counts, labels, iouv)
    res = ap_per_class_batched(det, counts, correct, labels, 80)
    cls = np.flatnonzero(res.present.cpu().numpy())
    assert np.array_equal(cls, g["seam/cls"]) and np.array_equal(res.nt.cpu().numpy(), g["seam/nt"])
    ap = res.ap.cpu().numpy()[cls]
    assert np.array_equal(ap[:, 0], g["seam/ap50"]) and np.array_equal(ap.mean(1), g["seam/ap"])
    p, r = res.p.cpu().numpy()[cls], res.r.cpu().numpy()[cls]
    assert np.allclose(p, g["seam/p"], rtol=0, atol=TOL) and np.allclose(r, g["seam/r"], rtol=0, atol=TOL)
    any_tp = bool(correct.any())
    assert any_tp == bool(g["seam/any"])
    mp, mr, map50, map_ = (p.mean(), r.mean(), ap[:, 0].mean(), ap.mean(1).mean()) if any_tp else (0.0, 0.0, 0.0, 0.0)
    for got, key in ((mp, "mp"), (mr, "mr"), (map50, "map50"), (map_, "map")):
        assert abs(float(got) - float(g[f"seam/{key}"])) <= TOL, key

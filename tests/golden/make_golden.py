"""Generate the golden fixtures in tests/golden/ by running the REFERENCE ITSELF (a checkout of ultralytics/yolov3 @ 97b87b1,
imported unmodified through oracle/ref_shim.py) on seeded inputs, and assert that the CPU oracle (oracle/yolo_oracle.py)
agrees with it.

    python tests/golden/make_golden.py --reference <checkout> [iou nms loss loss_edges forward scale val tta seam]

The fixtures it writes are committed; the tests compare against them and never read the reference.

What is pinned (SURVEY.md Appendix D):
  forward_<model>.npz   Model.forward (fused and unfused) -> z, raw p_i, layer taps      (models/yolo.py:135-147, 89-123)
  nms_cases.npz         non_max_suppression outputs for a sweep + adversarial cases       (utils/general.py:630-750)
  loss_cases.npz        ComputeLoss loss / loss_items / dL/dp and build_targets           (utils/loss.py:131-244)
  loss_edge_cases.npz   the same on the fp32 boundaries of build_targets, nc 1/2, nl 2/5, na 6, hyps (see gen_loss_edges)
  iou_cases.npz         box_iou, bbox_iou(CIoU) values                                    (ultralytics, via shim)
  val_cases.npz         val.process_batch correct[N,10] on seeded detections / labels     (val.py:147-188)
  tta_cases.npz         Model.forward(x, augment=True) rows (scale / flip views merged)    (models/yolo.py:239-280)
  seam_cases.npz        detect.py / val.py loop pieces, smart_optimizer groups, letterbox (see gen_seam)
"""
from __future__ import annotations

import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT / "oracle"))
import ref_shim  # noqa: E402
import yolo_oracle as O  # noqa: E402

OUT = Path(__file__).resolve().parent
CFG = ROOT / "yolov3_b200" / "cfg"


def ref_model(name, params):
    from models.yolo import Model  # reference

    m = Model(str(ref_shim.REFERENCE_ROOT / "models" / f"{name}.yaml"))
    missing, unexpected = m.load_state_dict(params, strict=False)
    assert not unexpected, unexpected
    assert all("num_batches_tracked" in k for k in missing), missing
    # the reference's own anchors/stride bookkeeping must equal the oracle's
    det = m.model[-1]
    assert torch.equal(det.anchors, params[[k for k in params if k.endswith(".anchors")][0]])
    return m.eval()


def gen_forward():
    cases = {"yolov3-tiny": [(1, 64, 64), (2, 96, 128)], "yolov3": [(1, 64, 64), (2, 64, 96)], "yolov3-spp": [(1, 64, 64)]}
    taps_for = {"yolov3": [0, 1, 6, 8, 15, 18, 22, 27], "yolov3-spp": [12, 15, 27], "yolov3-tiny": [0, 8, 12, 15, 18, 19]}
    for name, shapes in cases.items():
        params = O.init_params(CFG / f"{name}.yaml", seed=0)
        m = ref_model(name, params)
        store = {}
        for ci, (bs, h, w) in enumerate(shapes):
            x = torch.rand(bs, 3, h, w, generator=torch.Generator().manual_seed(100 + ci))
            # --- reference, unfused (BN in eval mode with running stats)
            feats = {}
            hooks = [m.model[i].register_forward_hook(lambda mod, inp, out, i=i: feats.__setitem__(i, out.detach().clone()))
                     for i in taps_for[name]]
            with torch.no_grad():
                z_ref, raw_ref = m(x.clone())
            for hk in hooks:
                hk.remove()
            # --- oracle, unfused and fused
            for fused in (False, True):
                om = O.OracleModel(CFG / f"{name}.yaml", params=params, fused=fused)
                taps = {i: None for i in taps_for[name]}
                with torch.no_grad():
                    z, raw = om(x.clone(), taps)
                tol = dict(atol=2e-4, rtol=2e-4) if fused else dict(atol=1e-5, rtol=1e-5)
                assert torch.allclose(z, z_ref, **tol), (name, fused, (z - z_ref).abs().max())
                for a, b in zip(raw, raw_ref):
                    assert torch.allclose(a, b, **tol), (name, fused, (a - b).abs().max())
                for i in taps:
                    assert torch.allclose(taps[i], feats[i], **tol), (name, i, fused)
            # --- reference fused (yolo.py:163-172) for completeness
            import copy

            mf = copy.deepcopy(m).fuse()
            with torch.no_grad():
                z_f, _ = mf(x.clone())
            assert torch.allclose(z_f, z_ref, atol=2e-4, rtol=2e-4)
            store[f"x{ci}_shape"] = np.array([bs, 3, h, w])
            store[f"x{ci}_seed"] = np.array(100 + ci)
            store[f"z{ci}"] = z_ref.numpy()
            for li, r in enumerate(raw_ref):
                store[f"raw{ci}_{li}"] = r.numpy()
            for i, t in feats.items():
                flat = t.flatten()
                idx = torch.linspace(0, flat.numel() - 1, 64).long()
                store[f"tap{ci}_{i}"] = np.concatenate([[t.mean().item(), t.std().item(), t.abs().max().item()], flat[idx].numpy()])
        store["param_seed"] = np.array(0)
        store["stride"] = m.stride.numpy()
        store["save"] = np.array(m.save)
        np.savez_compressed(OUT / f"forward_{name}.npz", **store)
        print("forward", name, "ok")


def nms_case_list():
    """(name, builder) -> prediction tensor [bs,n,85] and kwargs."""
    cases = []
    base = O.synth_predictions(2, n_rows=700, nc=80, seed=3)
    for ct, it in [(0.001, 0.6), (0.01, 0.6), (0.05, 0.45), (0.1, 0.45), (0.25, 0.45)]:
        for ml in (False, True):
            cases.append((f"sweep_c{ct}_ml{int(ml)}", base, dict(conf_thres=ct, iou_thres=it, multi_label=ml, max_det=300)))
    cases.append(("agnostic", base, dict(conf_thres=0.05, iou_thres=0.45, agnostic=True)))
    cases.append(("classes", base, dict(conf_thres=0.05, iou_thres=0.45, classes=[0, 3, 79])))
    cases.append(("maxdet1", base, dict(conf_thres=0.05, iou_thres=0.45, max_det=1)))
    cases.append(("maxdet1000", base, dict(conf_thres=0.001, iou_thres=0.6, max_det=1000, multi_label=True)))
    cases.append(("empty", base, dict(conf_thres=1.0, iou_thres=0.45)))
    # autolabel priors (general.py:689-695), (cls, x, y, w, h) rows in pixels.  Every prior has conf exactly 1.0 and the
    # reference's argsort is unstable, so the goldens carry at most one prior per image (tie-free, SURVEY App. C.3)
    cases.append(("labels", base, dict(conf_thres=0.25, iou_thres=0.45, labels=[[[3.0, 320.0, 320.0, 120.0, 90.0]], []])))
    cases.append(("labels_ml", base, dict(conf_thres=0.05, iou_thres=0.45, multi_label=True,
                                          labels=[[[3.0, 320.0, 320.0, 120.0, 90.0]], [[17.0, 100.5, 200.25, 50.0, 60.0]]])))
    # adversarial: zero-area boxes, identical boxes, class 0 and 79 with IoU near the threshold, fp16-rounded values
    g = torch.Generator().manual_seed(7)
    adv = torch.zeros(1, 64, 85)
    adv[0, :, 0:2] = torch.rand(64, 2, generator=g) * 40 + 300
    adv[0, :, 2:4] = torch.rand(64, 2, generator=g) * 60 + 20
    adv[0, :, 4] = torch.linspace(0.99, 0.5, 64)
    adv[0, :32, 5 + 0] = 0.9
    adv[0, 32:, 5 + 79] = 0.9
    adv[0, 5, 2:4] = 0.0  # zero-area box
    adv[0, 6, 2:4] = 0.0
    adv[0, 6, 0:2] = adv[0, 5, 0:2]  # two identical zero-area boxes: IoU = 0/0 = NaN -> both kept
    adv[0, 40, :4] = adv[0, 33, :4]  # identical boxes, class 79 (offset rounding) -> IoU 1 -> suppressed
    cases.append(("adversarial", adv, dict(conf_thres=0.25, iou_thres=0.45)))
    half = base.half().float()
    cases.append(("fp16_rounded", half, dict(conf_thres=0.05, iou_thres=0.45)))
    many = O.synth_predictions(1, n_rows=400, nc=80, seed=11)
    many[..., 4] = many[..., 4] * 0.5 + 0.5
    many[..., 5:] = many[..., 5:] * 0.5 + 0.5
    cases.append(("over_max_nms", many, dict(conf_thres=0.25, iou_thres=0.6, multi_label=True, max_det=300)))  # 32000 > 30000
    return cases


def gen_nms():
    import utils.general as G  # reference

    store, preds = {}, {}
    for name, pred, kw in nms_case_list():
        real_time = G.time.time
        G.time.time = lambda: 0.0  # disable the wall-clock time_limit break (utils/general.py:675,746-748)
        try:
            kw_ref = dict(kw)
            if "labels" in kw:  # the reference indexes label tensors
                kw_ref["labels"] = [torch.tensor(l, dtype=torch.float32).reshape(-1, 5) for l in kw["labels"]]
            ref = G.non_max_suppression(pred.clone(), **kw_ref)
        finally:
            G.time.time = real_time
        ora, src = O.non_max_suppression(pred.clone(), **kw)
        for xi, (r, o) in enumerate(zip(ref, ora)):
            r = r.numpy()
            assert r.shape == o.shape, (name, xi, r.shape, o.shape)
            assert np.array_equal(r, o), (name, xi, np.abs(r - o).max())
            store[f"{name}/out{xi}"] = r
            store[f"{name}/src{xi}"] = src[xi]
        pkey = preds.setdefault(id(pred), f"pred{len(preds)}")
        store[pkey] = pred.numpy().astype(np.float32)
        store[f"{name}/pred_key"] = np.array(pkey)
        store[f"{name}/kw"] = np.array(repr(kw))
        print("nms", name, [len(r) for r in ref])
    np.savez_compressed(OUT / "nms_cases.npz", **store)


SCALE_CASES = [((640, 640), (1080, 810, 3), None), ((384, 640), (720, 1280, 3), None), ((640, 480), (375, 500, 3), None),
               ((640, 640), (480, 640, 3), ((0.75, 0.75), (16.0, 80.0)))]


def gen_scale_boxes():
    """scale_boxes (utils/general.py:613-626, through the shim's clip_boxes) on seeded xyxy boxes incl. out-of-image ones."""
    import utils.general as G  # reference

    store = {}
    for ci, (s1, s0, rp) in enumerate(SCALE_CASES):
        g = torch.Generator().manual_seed(40 + ci)
        xy = torch.rand(200, 2, generator=g) * torch.tensor([s1[1], s1[0]]) * 1.2 - 0.1 * torch.tensor([s1[1], s1[0]])
        wh = torch.rand(200, 2, generator=g) * 300
        boxes = torch.cat((xy - wh / 2, xy + wh / 2, torch.rand(200, 2, generator=g)), 1)  # [200, 6] like the NMS output
        ref = boxes.clone()
        G.scale_boxes(s1, ref[:, :4], s0, rp)
        ora = O.scale_boxes(s1, boxes[:, :4].numpy(), s0, rp)
        assert np.array_equal(ref[:, :4].numpy(), ora), (ci, np.abs(ref[:, :4].numpy() - ora).max())
        store[f"in{ci}"] = boxes.numpy()
        store[f"out{ci}"] = ref.numpy()
        store[f"geom{ci}"] = np.array(repr((s1, s0, rp)))  # (img1_shape, img0_shape, ratio_pad) for the tests
    np.savez_compressed(OUT / "scale_boxes_cases.npz", **store)
    print("scale_boxes ok")


def loss_inputs(case):
    g = torch.Generator().manual_seed(200 + case)
    bs = [2, 3, 1, 2][case]
    hw = [(8, 8), (8, 12), (4, 4), (8, 8)][case]
    p = [torch.randn(bs, 3, hw[0] * s, hw[1] * s, 85, generator=g) for s in (4, 2, 1)]
    if case == 0:
        t = O.synth_targets(bs, seed=2)
    elif case == 1:
        t = O.synth_targets(bs, seed=5)
        t[0, 2:4] = torch.tensor([0.5, 0.5])  # exactly on a cell border at every level
        t[1, 2:4] = torch.tensor([0.001, 0.999])  # near the image edge -> index clamp
    elif case == 2:
        t = torch.zeros(0, 6)  # no targets
    else:
        t = O.synth_targets(bs, seed=9)[:1]  # single target
    return p, t


def gen_loss():
    from utils.loss import ComputeLoss  # reference

    name = "yolov3"
    params = O.init_params(CFG / f"{name}.yaml", seed=0)
    m = ref_model(name, params)
    m.hyp = O.scaled_hyp()
    cl = ComputeLoss(m)
    anchors = m.model[-1].anchors
    store = {"hyp": np.array(repr(m.hyp))}
    for case in range(4):
        p, t = loss_inputs(case)
        pr = [x.clone().requires_grad_(True) for x in p]
        loss, items = cl(pr, t.clone())
        loss.backward()
        po = [x.clone().requires_grad_(True) for x in p]
        lo, io = O.compute_loss(po, t.clone(), anchors, m.hyp)
        lo.backward()
        assert torch.allclose(loss, lo, rtol=1e-5, atol=1e-6), (case, loss, lo)
        assert torch.allclose(items, io, rtol=1e-5, atol=1e-6)
        for a, b in zip(pr, po):
            assert torch.allclose(a.grad, b.grad, rtol=1e-4, atol=1e-7), (case, (a.grad - b.grad).abs().max())
        # build_targets
        tcls, tbox, indices, anch = cl.build_targets(pr, t.clone())
        bt = O.build_targets([tuple(x.shape) for x in p], t, anchors, m.hyp["anchor_t"])
        for i in range(3):
            assert torch.equal(tcls[i], bt[i]["tcls"]) and torch.allclose(tbox[i], bt[i]["tbox"])
            for a, k in zip(indices[i], ("b", "a", "gj", "gi")):
                assert torch.equal(a, bt[i][k]), (case, i, k)
            assert torch.equal(anch[i], bt[i]["anch"])
            store[f"c{case}/bt{i}"] = torch.cat(
                (torch.stack([x.float() for x in indices[i]], 1), tbox[i], anch[i], tcls[i][:, None].float()), 1).numpy()
        store[f"c{case}/loss"] = loss.detach().numpy()
        store[f"c{case}/items"] = items.numpy()
        for i, a in enumerate(pr):
            store[f"c{case}/grad{i}"] = a.grad.numpy()
        store[f"c{case}/targets"] = t.numpy()
        print("loss", case, float(loss), items.tolist())
    store["anchors"] = anchors.numpy()
    np.savez_compressed(OUT / "loss_cases.npz", **store)


# ---------------------------------------------------------------------------------------------------------------------- loss edges
# Anchors in pixels per level, as in the model yamls; divided by the stride they are the grid units the loss sees.
ANCHORS_PX = {
    "yolov3": (((10, 13), (16, 30), (33, 23)), ((30, 61), (62, 45), (59, 119)), ((116, 90), (156, 198), (373, 326))),
    "yolov3-tiny": (((10, 14), (23, 27), (37, 58)), ((81, 82), (135, 169), (344, 319))),
    # the ABI maxima: 5 levels x 6 anchors (P3-P7), growing 1.5x per level so that small images match on every level
    "p3p7x6": tuple(tuple((round(w * 1.5**l), round(h * 1.5**l)) for w, h in ((10, 13), (16, 30), (33, 23), (30, 61),
                                                                              (62, 45), (59, 119))) for l in range(5)),
}
STRIDES = {"yolov3": (8, 16, 32), "yolov3-tiny": (16, 32), "p3p7x6": (8, 16, 32, 64, 128)}


def grid_anchors(kind):
    return torch.tensor(ANCHORS_PX[kind], dtype=torch.float32) / torch.tensor(STRIDES[kind], dtype=torch.float32)[:, None, None]


def f32(v):
    return np.float32(v)


def f32_preimage(fn, want, start, span=256):
    """The float32 x nearest to `start` with fn(x) == want (fn evaluated in float32), searched over +-span ulps."""
    x0 = f32(start)
    up, down = x0, x0
    for _ in range(span):
        for x in (up, down):
            if fn(x) == f32(want):
                return x
        up, down = np.nextafter(up, f32(np.inf)), np.nextafter(down, f32(-np.inf))
    raise AssertionError(f"no float32 preimage of {want} near {start}")


def f32_straddle(fn, want, start, span=4096):
    """Adjacent float32 inputs a < b near `start` with fn(a) < want <= fn(b) or fn(a) >= want > fn(b) (fn in float32)."""
    x = f32(start)
    below = fn(x) < f32(want)
    for to in (f32(np.inf), f32(-np.inf)):
        v = x
        for _ in range(span):
            n = np.nextafter(v, to)
            if (fn(n) < f32(want)) != below:
                return (v, n) if to > 0 else (n, v)
            v = n
    raise AssertionError(f"fn does not cross {want} near {start}")


def f32_neighbours(fn, x):
    """The float32 inputs nearest to x, below and above, at which fn (evaluated in float32) takes a different value."""
    out = []
    for to in (f32(-np.inf), f32(np.inf)):
        v = x
        while fn(v) == fn(x):
            v = np.nextafter(v, to)
        out.append(v)
    return tuple(out)


def edge_targets(family, kind, imgsz, nc=80, bs=2, anchor_t=4.0):
    """Target rows [nt, 6] (img, cls, x, y, w, h) that sit on the fp32 boundaries of build_targets (utils/loss.py:207-240)
    for the grids of `kind` at image size `imgsz` = (h, w).  Boxes are 40 px unless the family needs otherwise: the wh
    ratio to an anchor does not depend on the level (w * imgsz / anchor_px), and 40 px passes anchor_t = 4 on every level
    of yolov3, so a centre on the image edge is matched, and clamped, on every level."""
    H, W = imgsz
    grids = [(H // s, W // s) for s in STRIDES[kind]]
    bw, bh = f32(40 / W), f32(40 / H)
    rows = []

    def row(b, c, x, y, w=bw, h=bh):
        rows.append([b, c % nc, x, y, w, h])

    if family == "image_edge":
        for b in range(bs):
            for k, (x, y) in enumerate([(0.0, 0.0), (1.0, 1.0), (0.0, 1.0), (1.0, 0.0), (0.4, 1.0), (1.0, 0.4),
                                        (0.0, 0.55), (0.7, 0.0)]):
                row(b, 3 + k + b, x, y)
    elif family == "cell_borders":
        ks = (1, 2, 3, 4, 6, 8, 13, 16, 22, 32, 37, 48, 58, 60, 62, 63)  # x, y = k / 64: gxy % 1 lands on 0, .25, .5, .75
        for i, kx in enumerate(ks):
            row(i % bs, i, kx / 64, ks[(i * 7 + 3) % len(ks)] / 64)
        for ny, nx in grids:  # gxy == 1.0 and gxi == n - gxy == 1.0 exactly, which the strict '> 1' rejects
            x1 = f32_preimage(lambda v: v * f32(nx), 1.0, 1.0 / nx)
            y1 = f32_preimage(lambda v: v * f32(ny), 1.0, 1.0 / ny)
            xn = f32_preimage(lambda v: f32(nx) - v * f32(nx), 1.0, (nx - 1.0) / nx)
            yn = f32_preimage(lambda v: f32(ny) - v * f32(ny), 1.0, (ny - 1.0) / ny)
            xh = f32_preimage(lambda v: v * f32(nx), nx // 2 + 0.5, (nx // 2 + 0.5) / nx)  # gxy % 1 == 0.5 exactly
            for b, (x, y) in enumerate([(x1, y1), (xn, yn), (x1, yn), (xh, 0.5), (0.5, y1)]):
                row(b % bs, 7 * b + nx, x, y)
    elif family == "anchor_ratio":
        t = f32(anchor_t)
        anchors = grid_anchors(kind).numpy()
        for l, (ny, nx) in enumerate(grids):
            a = (l * 2 + 1) % anchors.shape[1]
            aw, ah = anchors[l, a]
            h = f32(ah / f32(ny))  # gh / ah == 1: the w side decides
            r_side = lambda v: (v * f32(nx)) / aw  # noqa: E731
            inv_side = lambda v: f32(1) / ((v * f32(nx)) / aw)  # noqa: E731
            for side, (fn, start) in enumerate(((r_side, float(t) * aw / nx), (inv_side, aw / (float(t) * nx)))):
                # the two fp32 inputs whose ratios straddle anchor_t; where one of them is exactly anchor_t (rejected), also
                # the nearest ratios either side of it that fp32 can reach
                ws = list(f32_straddle(fn, t, start))
                ws += [v for w in ws if fn(w) == t for v in f32_neighbours(fn, w)]
                for v in ws:
                    row(l % bs, 10 * l + side, 0.3 + 0.1 * l, 0.6 - 0.2 * side, v, h)
    elif family == "shared_cells":
        x, y = 0.3 + 1 / 256, 0.6 + 1 / 256  # inside one cell on every level, away from the cell borders
        row(0, 5, x, y)
        row(0, 5, x, y)  # the same target twice
        row(0, 7, x + 1 / 1024, y, bw * 1.1)  # same cell, different class
        row(0, 9, x - 1 / 1024, y + 1 / 1024, bw * 0.95, bh * 1.05)  # >= 3 matches on the cell (and on its neighbours)
        gx0 = grids[0][1]
        row(1, 11, (3 + 0.25) / gx0, 0.5 + 0.25 / grids[0][0])  # frac .25 -> also matched one cell to the left ...
        row(1, 12, (2 + 0.6) / gx0, 0.5 + 0.25 / grids[0][0], bw * 1.2)  # ... which is this target's own cell
    else:
        raise KeyError(family)
    return torch.tensor(rows, dtype=torch.float32).reshape(-1, 6)


def random_targets(bs, nc, seed, per_image=6, empty=()):
    """synth_targets-like rows with a given number of targets per image; images in `empty` get none."""
    g = torch.Generator().manual_seed(seed)
    t = O.synth_targets(bs, nc=nc, seed=seed)
    keep = torch.tensor([int(b) not in empty for b in t[:, 0].tolist()], dtype=torch.bool)
    t = t[keep]
    return t[torch.randperm(len(t), generator=g)[: per_image * bs]] if per_image else t


def loss_edge_case_list():
    """(name, spec) for loss_edge_cases.npz.  spec: kind (anchor set), imgsz (h, w), bs, nc, hyp overrides, targets builder,
    logit saturation.  Small images, so that repeated writes to a cell stay few and the reference's tobj is well defined."""
    return [
        ("image_edge", dict(kind="yolov3", imgsz=(128, 128), bs=2, nc=80, fam="image_edge")),
        ("image_edge_rect", dict(kind="yolov3", imgsz=(96, 160), bs=2, nc=80, fam="image_edge")),
        ("cell_borders", dict(kind="yolov3", imgsz=(128, 128), bs=2, nc=80, fam="cell_borders")),
        ("cell_borders_640", dict(kind="yolov3", imgsz=(640, 640), bs=1, nc=4, fam="cell_borders")),
        ("anchor_ratio", dict(kind="yolov3", imgsz=(128, 128), bs=3, nc=80, fam="anchor_ratio")),
        ("anchor_ratio_t291", dict(kind="yolov3", imgsz=(128, 128), bs=3, nc=80, fam="anchor_ratio", hyp=dict(anchor_t=2.91))),
        ("shared_cells", dict(kind="yolov3", imgsz=(128, 128), bs=2, nc=80, fam="shared_cells")),
        ("nc1_smoothing", dict(kind="yolov3", imgsz=(128, 128), bs=2, nc=1, fam="random",
                               hyp=dict(label_smoothing=0.1, obj_pw=1.3))),
        ("nc2_hyps", dict(kind="yolov3", imgsz=(128, 128), bs=2, nc=2, fam="random",
                          hyp=dict(label_smoothing=0.1, cls_pw=1.7, obj_pw=0.6))),
        ("tiny_nl2", dict(kind="yolov3-tiny", imgsz=(128, 96), bs=2, nc=80, fam="random")),
        ("abi_max_nl5_na6", dict(kind="p3p7x6", imgsz=(256, 256), bs=1, nc=6, fam="random")),
        ("rect_empty_images", dict(kind="yolov3", imgsz=(96, 160), bs=3, nc=80, fam="random", empty=(1,))),
        ("saturated", dict(kind="yolov3", imgsz=(128, 128), bs=2, nc=80, fam="random", sat=12.0)),
    ]


def loss_edge_inputs(spec, seed):
    """(p list, targets, anchors [nl, na, 2] grid units, hyp) for one edge case."""
    kind, (H, W), bs, nc = spec["kind"], spec["imgsz"], spec["bs"], spec["nc"]
    hyp = O.scaled_hyp(nl=len(STRIDES[kind]), nc=nc, imgsz=max(H, W))
    hyp.update(spec.get("hyp", {}))
    if spec["fam"] == "random":
        t = random_targets(bs, nc, seed, per_image=4, empty=spec.get("empty", ()))
    else:
        t = edge_targets(spec["fam"], kind, (H, W), nc=nc, bs=bs, anchor_t=hyp["anchor_t"])
    anchors = grid_anchors(kind)
    g = torch.Generator().manual_seed(300 + seed)
    p = [torch.randn(bs, anchors.shape[1], H // s, W // s, nc + 5, generator=g) for s in STRIDES[kind]]
    if spec.get("sat"):  # logits at +-sat: each entry's sign drawn at random (tw/th pushed to -sat would underflow pwh)
        for x in p:
            sgn = torch.where(torch.rand(x.shape, generator=g) < 0.5, -1.0, 1.0)
            x.copy_(torch.where(torch.rand(x.shape, generator=g) < 0.5, sgn * spec["sat"], x))
            x[..., 2:4] = x[..., 2:4].abs().clamp(max=3.0)  # pwh = (2 sigmoid)^2 anchor stays away from 0 (0/0 in CIoU)
    return p, t, anchors, hyp


class _RefLossModel(torch.nn.Module):
    """What the reference's ComputeLoss reads from a model: a parameter (for the device), .hyp and model[-1] = Detect."""

    def __init__(self, anchors, nc, strides, hyp):
        super().__init__()
        from types import SimpleNamespace

        self.w = torch.nn.Parameter(torch.zeros(1))
        self.hyp = hyp
        self.model = [SimpleNamespace(nl=anchors.shape[0], na=anchors.shape[1], nc=nc, anchors=anchors,
                                      stride=torch.tensor(strides, dtype=torch.float32))]


def gen_loss_edges():
    """loss_edge_cases.npz: the reference's ComputeLoss on the fp32 boundaries of build_targets, asserted against the oracle."""
    from utils.loss import ComputeLoss  # reference

    store = {}
    for ci, (name, spec) in enumerate(loss_edge_case_list()):
        p, t, anchors, hyp = loss_edge_inputs(spec, ci)
        nc = spec["nc"]
        cl = ComputeLoss(_RefLossModel(anchors, nc, STRIDES[spec["kind"]], hyp))
        pr = [x.clone().requires_grad_(True) for x in p]
        loss, items = cl(pr, t.clone())
        loss.backward()
        po = [x.clone().requires_grad_(True) for x in p]
        lo, io = O.compute_loss(po, t.clone(), anchors, hyp, nc=nc)
        lo.backward()
        assert torch.allclose(loss, lo, rtol=1e-5, atol=1e-6), (name, loss, lo)
        assert torch.allclose(items, io, rtol=1e-5, atol=1e-6), (name, items, io)
        for a, b in zip(pr, po):
            assert torch.allclose(a.grad, b.grad, rtol=1e-4, atol=1e-7), (name, (a.grad - b.grad).abs().max())
        tcls, tbox, indices, anch = cl.build_targets(pr, t.clone())
        bt = O.build_targets([tuple(x.shape) for x in p], t, anchors, hyp["anchor_t"])
        for i in range(len(p)):
            assert torch.equal(tcls[i], bt[i]["tcls"]) and torch.allclose(tbox[i], bt[i]["tbox"]), (name, i)
            for a, k in zip(indices[i], ("b", "a", "gj", "gi")):
                assert torch.equal(a, bt[i][k]), (name, i, k)
            assert torch.equal(anch[i], bt[i]["anch"])
            store[f"{name}/bt{i}"] = torch.cat(
                (torch.stack([x.float() for x in indices[i]], 1), tbox[i], anch[i], tcls[i][:, None].float()), 1).numpy()
        store[f"{name}/loss"], store[f"{name}/items"] = loss.detach().numpy(), items.numpy()
        for i, a in enumerate(pr):
            store[f"{name}/grad{i}"] = a.grad.numpy()
        store[f"{name}/targets"], store[f"{name}/hyp"] = t.numpy(), np.array(repr(hyp))
        store[f"{name}/seed"] = np.array(ci)
        print("loss_edges", name, len(t), "targets", [len(x) for x in tcls], "matches", float(loss), items.tolist())
    store["cases"] = np.array([n for n, _ in loss_edge_case_list()])
    np.savez_compressed(OUT / "loss_edge_cases.npz", **store)


def gen_iou():
    from utils.metrics import box_iou  # reference re-export (shim restatement of the ultralytics formula)
    import torchvision

    g = torch.Generator().manual_seed(5)
    a = torch.rand(40, 4, generator=g) * 300
    a[:, 2:] += a[:, :2]
    b = torch.rand(25, 4, generator=g) * 300
    b[:, 2:] += b[:, :2]
    b[0] = a[0]
    b[1, 2:] = b[1, :2]  # zero-area
    r = box_iou(a, b)
    assert torch.allclose(r, torchvision.ops.box_iou(a, b), atol=1e-6)
    assert torch.allclose(r, O.box_iou(a, b), atol=0, rtol=0)
    # CIoU vs float64 restatement
    p1 = torch.rand(64, 4, generator=g) * 4 + 0.1
    p2 = torch.rand(64, 4, generator=g) * 4 + 0.1
    from ultralytics.utils.metrics import bbox_iou

    c32 = bbox_iou(p1, p2, CIoU=True).squeeze()
    c64 = O.ciou_xywh(p1.double(), p2.double())
    assert torch.allclose(c32.double(), c64, atol=1e-5)
    assert torch.allclose(c32, O.ciou_xywh(p1, p2), atol=1e-6)
    np.savez_compressed(OUT / "iou_cases.npz", a=a.numpy(), b=b.numpy(), iou=r.numpy(), p1=p1.numpy(), p2=p2.numpy(),
                        ciou=c32.numpy())
    print("iou ok")


def gen_tta():
    """Model.forward(x, augment=True) (models/yolo.py:233-280) of the reference vs the oracle restatement."""
    store = {}
    for name, shape in (("yolov3-tiny", (2, 3, 96, 128)), ("yolov3", (1, 3, 128, 96))):
        params = O.init_params(CFG / f"{name}.yaml", seed=0)
        m = ref_model(name, params)
        x = torch.rand(*shape, generator=torch.Generator().manual_seed(41))
        with torch.no_grad():
            z_ref = m(x.clone(), augment=True)[0]
            z_ora = O.forward_augment(O.OracleModel(CFG / f"{name}.yaml", params=params, fused=False), x)
        assert z_ref.shape == z_ora.shape, (z_ref.shape, z_ora.shape)
        err = float((z_ref - z_ora).abs().max() / z_ref.abs().max())
        assert err < 2e-5, (name, err)
        store[f"{name}/shape"], store[f"{name}/z_aug"] = np.array(shape), z_ref.numpy().astype(np.float32)
        print("tta", name, tuple(z_ref.shape), err)
    np.savez_compressed(OUT / "tta_cases.npz", **store)


def val_case_list():
    """(name, n_det, n_lab, nc, seed, jitter): crowded / sparse / empty-side / single-pair / many-duplicates cases"""
    return [("typical", 120, 25, 6, 0, 12.0), ("crowded", 300, 60, 3, 1, 6.0), ("sparse", 40, 5, 20, 2, 25.0),
            ("one_pair", 1, 1, 1, 3, 1.0), ("no_labels", 30, 0, 4, 4, 5.0), ("one_label_many_dets", 80, 1, 1, 5, 4.0),
            ("many_labels_one_det", 1, 40, 2, 6, 8.0), ("tight", 200, 30, 2, 7, 2.0)]


def gen_val():
    import val as V  # reference val.py (process_batch)

    iouv = torch.linspace(0.5, 0.95, 10)  # val.py:301
    store = {"iouv": iouv.numpy()}
    for name, nd, nl, nc, seed, jit in val_case_list():
        det, lab = O.synth_val_case(nd, nl, nc, seed, jit)
        if nl == 0:
            ref = torch.zeros(nd, 10, dtype=torch.bool)  # val.py:372-376 never calls process_batch without labels
        else:
            ref = V.process_batch(det, lab, iouv)
        ora = O.process_batch(det, lab, iouv) if nl else ref
        assert torch.equal(ref, ora), name
        store[f"{name}/det"], store[f"{name}/lab"], store[f"{name}/correct"] = det.numpy(), lab.numpy(), ref.numpy()
        print("val", name, int(ref.sum()), "true of", ref.numel())
    np.savez_compressed(OUT / "val_cases.npz", **store)


SEAM_IMGSZ = 128  # detect.py's image size for the seam fixture: small enough to store its inputs and predictions
LETTERBOX_SHAPES = [(1080, 810), (375, 500), (333, 1000)]
LETTERBOX_KW = [dict(auto=True), dict(auto=False), dict(auto=False, scaleFill=True), dict(auto=True, scaleup=False)]


def gen_seam():
    """What the seam tests (tests/test_zz_reference_seam_gpu.py, tests/test_params_cpu.py, tests/test_oracle_golden.py)
    compare against:
      detect/<i>/*     detect.py:166-223 on data/images with yolov3-tiny (confident weights): LoadImages' letterboxed input,
                       Model forward z, non_max_suppression(0.25, 0.45, max_det=50), scale_boxes to the native image
      val/<si>/*       val.py:355-390 on synthetic predictions: NMS(0.001, 0.6, multi-label), scale_boxes, process_batch
      optim/<cfg>/<g>  smart_optimizer(SGD, 0.01, 0.937, 5e-4) (utils/torch_utils.py:207-237): parameter names per group and
                       (lr, momentum, dampening, weight_decay, nesterov)
      letterbox/<i>_<k>  utils/augmentations.py letterbox on seeded random images: sha256 of the image, ratio, pad"""
    import hashlib

    import utils.general as G  # reference
    import val as V  # reference
    from models.yolo import Model  # reference
    from utils.augmentations import letterbox  # reference
    from utils.dataloaders import LoadImages  # reference
    from utils.torch_utils import smart_optimizer  # reference

    sys.path.insert(0, str(ROOT))
    from yolov3_b200.module import DetectionModel

    store = {}
    real_time = G.time.time
    G.time.time = lambda: 0.0  # disable the wall-clock time_limit break (utils/general.py:675,746-748)
    try:
        params = O.confident_params(CFG / "yolov3-tiny.yaml")
        m = ref_model("yolov3-tiny", params)
        images = LoadImages(str(ref_shim.REFERENCE_ROOT / "data" / "images"), img_size=(SEAM_IMGSZ, SEAM_IMGSZ), stride=32, auto=True)
        for i, (path, im, im0s, _, _) in enumerate(images):
            x = torch.from_numpy(im).float()[None] / 255
            with torch.no_grad():
                z = m(x)[0]
            det = G.non_max_suppression(z.clone(), 0.25, 0.45, max_det=50)[0]
            assert len(det) >= 1, path
            # bit-equal confidences are ordered by an unstable argsort in the reference and by index in the oracle (and in
            # yolov3_b200): the fixture must not depend on that order, i.e. both keep the same set of rows
            (ora,), _ = O.non_max_suppression(z.clone(), 0.25, 0.45, max_det=50)
            a = det.numpy()
            assert np.array_equal(a[np.lexsort(a.T[::-1])], ora[np.lexsort(ora.T[::-1])]), path
            store[f"detect/{i}/im"], store[f"detect/{i}/im0_shape"] = im, np.array(im0s.shape)
            store[f"detect/{i}/z"], store[f"detect/{i}/det"] = z.numpy(), a
            store[f"detect/{i}/scaled"] = G.scale_boxes(x.shape[2:], det[:, :4].clone(), im0s.shape).numpy()
            print("seam detect", Path(path).name, tuple(im.shape), len(det))

        pred = O.synth_predictions(2, n_rows=3000, nc=80, seed=5)
        targets = O.synth_targets(2, seed=4)
        h = w = 640
        shape0, ratio_pad = (480, 600), ((1.0667, 1.0667), (0.0, 64.0))
        targets[:, 2:] *= torch.tensor((w, h, w, h))
        iouv = torch.linspace(0.5, 0.95, 10)
        out = G.non_max_suppression(pred.clone(), 0.001, 0.6, multi_label=True, max_det=300)
        for si in range(2):
            labels = targets[targets[:, 0] == si, 1:]
            predn = out[si].clone()
            G.scale_boxes((h, w), predn[:, :4], shape0, ratio_pad)
            tbox = G.xywh2xyxy(labels[:, 1:5])
            G.scale_boxes((h, w), tbox, shape0, ratio_pad)
            labelsn = torch.cat((labels[:, 0:1], tbox), 1)
            store[f"val/{si}/out"], store[f"val/{si}/predn"] = out[si].numpy(), predn.numpy()
            store[f"val/{si}/labelsn"], store[f"val/{si}/correct"] = labelsn.numpy(), V.process_batch(predn, labelsn, iouv).numpy()
    finally:
        G.time.time = real_time

    for name in ("yolov3", "yolov3-tiny"):
        groups = []
        for model in (Model(str(ref_shim.REFERENCE_ROOT / "models" / f"{name}.yaml")), DetectionModel(CFG / f"{name}.yaml", device="cpu")):
            by_ptr = {p.data_ptr(): n for n, p in model.named_parameters()}
            opt = smart_optimizer(model, "SGD", 0.01, 0.937, 5e-4)
            groups.append([(sorted(by_ptr[p.data_ptr()] for p in g["params"]),
                            [g["lr"], g["momentum"], g["dampening"], g["weight_decay"], float(g["nesterov"])]) for g in opt.param_groups])
        assert groups[0] == groups[1], name  # the reference's own Model and the nn.Module facade group alike
        for gi, (names, hyp) in enumerate(groups[0]):
            store[f"optim/{name}/{gi}/names"], store[f"optim/{name}/{gi}/hyp"] = np.array(names), np.array(hyp)
        print("seam optim", name, [len(n) for n, _ in groups[0]])

    rng = np.random.default_rng(1)
    store["letterbox/shapes"], store["letterbox/kw"] = np.array(LETTERBOX_SHAPES), np.array(repr(LETTERBOX_KW))
    for i, (h, w) in enumerate(LETTERBOX_SHAPES):
        im = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        for k, kw in enumerate(LETTERBOX_KW):
            a = letterbox(im.copy(), **kw)
            store[f"letterbox/{i}_{k}/sha256"] = np.array(hashlib.sha256(np.ascontiguousarray(a[0]).tobytes()).hexdigest())
            store[f"letterbox/{i}_{k}/shape"] = np.array(a[0].shape)
            store[f"letterbox/{i}_{k}/ratio"], store[f"letterbox/{i}_{k}/pad"] = np.array(a[1], np.float64), np.array(a[2], np.float64)
    np.savez_compressed(OUT / "seam_cases.npz", **store)
    print("seam ok")


if __name__ == "__main__":
    args = sys.argv[1:]
    if "--reference" in args:
        i = args.index("--reference")
        ref_shim.REFERENCE_ROOT = Path(args[i + 1]).resolve()
        del args[i:i + 2]
    assert ref_shim.reference_available(), "pass --reference <checkout of ultralytics/yolov3 @ 97b87b1>"
    ref_shim.install()
    torch.set_num_threads(8)
    which = args or ["iou", "nms", "loss", "loss_edges", "forward", "scale", "val", "tta", "seam"]
    if "seam" in which:
        gen_seam()
    if "tta" in which:
        gen_tta()
    if "val" in which:
        gen_val()
    if "scale" in which:
        gen_scale_boxes()
    if "iou" in which:
        gen_iou()
    if "nms" in which:
        gen_nms()
    if "loss" in which:
        gen_loss()
    if "loss_edges" in which:
        gen_loss_edges()
    if "forward" in which:
        gen_forward()

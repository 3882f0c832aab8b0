"""y3_loss_fwd_bwd (csrc/y3_loss.cu) at the edges of build_targets, against the float64 restatement (tests/loss_oracle.py)
and the reference goldens of tests/golden/loss_edge_cases.npz.

Observables per case:
  - loss and loss_items: relative error <= 2e-5 against float64;
  - dL/dp per level: |g - ref| <= 1e-4 |ref| + 1e-6 max|ref|;
  - the matched-cell set: the cells with any nonzero gradient in slots 0-3 and 5+ equal the restatement's matches exactly,
    which checks build_targets' fp32 decisions independently of any tolerance;
  - the tobj winner: a second run with every objectness logit at 0 and obj_pw = 1 has d(loss)/d(p4) = k (0.5 - tobj) with
    k = obj * bs * balance / cells, so tobj per cell is read back from the gradient and compared with the restatement's;
    on a cell several matches share this shows which match won (the last in the reference's order).
"""
import ast
import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent))
sys.path.insert(0, str(Path(__file__).resolve().parent / "golden"))
import loss_oracle as LO  # noqa: E402
from make_golden import grid_anchors, loss_edge_case_list, loss_edge_inputs  # noqa: E402

pytestmark = pytest.mark.gpu
G = Path(__file__).parent / "golden"
EDGE = dict(loss_edge_case_list())


def _loss(anchors, nc, hyp):
    from yolov3_b200.loss import ComputeLoss

    det = SimpleNamespace(nl=anchors.shape[0], na=anchors.shape[1], nc=nc, anchors=anchors)
    return ComputeLoss(SimpleNamespace(model=[det], hyp=hyp))


def _kernel(p, t, anchors, hyp, upstream=1.0, grad=True):
    nc = p[0].shape[-1] - 5
    pc = [x.cuda().requires_grad_(grad) for x in p]
    loss, items = _loss(anchors, nc, hyp)(pc, t.cuda())
    if grad:
        (loss * upstream).backward()
    torch.cuda.synchronize()
    return (float(loss.detach()), items.cpu().numpy().astype(np.float64),
            [x.grad.cpu().numpy().astype(np.float64) for x in pc] if grad else None)


def _compare(p, t, anchors, hyp, t_ref=None):
    """Kernel vs restatement on every observable.  t_ref: the rows the restatement sees (default: t)."""
    r = LO.compute_loss(p, t if t_ref is None else t_ref, anchors, hyp)
    loss, items, grads = _kernel(p, t, anchors, hyp)
    assert abs(loss - r["loss"]) <= 2e-5 * abs(r["loss"]), (loss, r["loss"])
    assert np.all(np.abs(items - r["items"]) <= 2e-5 * np.abs(r["items"]) + 1e-9), (items, r["items"])
    nl, bs = len(p), p[0].shape[0]
    cells = set()
    for l in range(nl):
        g, ref = grads[l], r["grads"][l]
        bad = np.abs(g - ref) > 1e-4 * np.abs(ref) + 1e-6 * np.abs(ref).max()
        assert not bad.any(), (l, int(bad.sum()), np.abs(g - ref).max(), np.argwhere(bad)[:4])
        hit = (g[..., 0:4] != 0).any(-1) | (g[..., 5:] != 0).any(-1)
        cells |= {(l,) + tuple(c) for c in np.argwhere(hit).tolist()}
    assert cells == r["cells"], (sorted(cells - r["cells"])[:5], sorted(r["cells"] - cells)[:5])
    # the tobj each cell ended up with (the restatement's tobj does not depend on the objectness logits or on obj_pw)
    p0 = [x.clone() for x in p]
    for x in p0:
        x[..., 4] = 0.0
    h1 = dict(hyp, obj_pw=1.0)
    _, _, g0 = _kernel(p0, t, anchors, h1)
    bal = LO.balance_for(nl)
    for l in range(nl):
        k = hyp["obj"] * bs * bal[l] / np.prod(p[l].shape[:4])
        tobj = 0.5 - g0[l][..., 4] / k
        assert np.allclose(tobj, r["tobj"][l], rtol=0, atol=2e-5), (l, np.abs(tobj - r["tobj"][l]).max())
    return r


def _spec(kind="yolov3", imgsz=(640, 640), bs=2, nc=80, fam="random", **kw):
    return dict(kind=kind, imgsz=imgsz, bs=bs, nc=nc, fam=fam, **kw)


# ---------------------------------------------------------------------------------------------------------------------- families
FAMILIES = {
    "image_edge": _spec(fam="image_edge"),
    "image_edge_rect": _spec(imgsz=(384, 640), fam="image_edge"),
    "cell_borders": _spec(fam="cell_borders"),
    "cell_borders_rect": _spec(imgsz=(384, 640), bs=1, fam="cell_borders"),
    "anchor_ratio": _spec(bs=3, fam="anchor_ratio"),
    "anchor_ratio_t291": _spec(bs=3, fam="anchor_ratio", hyp=dict(anchor_t=2.91)),
    "shared_cells": _spec(fam="shared_cells"),
    "nc1": _spec(nc=1),
    "nc2": _spec(nc=2),
    "tiny_nl2": _spec(kind="yolov3-tiny", imgsz=(416, 416)),
    "abi_max_nl5_na6": _spec(kind="p3p7x6", nc=6),
    "rect_val_384x640": _spec(imgsz=(384, 640), bs=4, empty=(0, 2)),
    "label_smoothing_pw": _spec(hyp=dict(label_smoothing=0.1, cls_pw=1.7, obj_pw=0.6)),
    "saturated": _spec(sat=12.0),
}


@pytest.mark.parametrize("name", list(FAMILIES))
def test_loss_edges_vs_float64(name):
    p, t, anchors, hyp = loss_edge_inputs(FAMILIES[name], 50 + list(FAMILIES).index(name))
    r = _compare(p, t, anchors, hyp)
    assert sum(len(m["b"]) for m in r["matches"]) > 0


def test_image_edge_tbox_uses_clamped_cell():
    """A centre at x = 1.0 lies in the clamped cell nx - 1 with tbox x = 1.0 (the reference clamps gij in place before it
    forms gxy - gij).  The single-target case of the bug report: the kernel matches the restatement there."""
    anchors = grid_anchors("yolov3")
    hyp = LO_hyp()
    t = torch.tensor([[0, 3, 0.4, 1.0, 0.1, 0.1]])
    g = torch.Generator().manual_seed(7)
    p = [torch.randn(1, 3, n, n, 85, generator=g) for n in (32, 16, 8)]
    r = _compare(p, t, anchors, hyp)
    assert any((m["tbox"][:, 1] == 1.0).any() for m in r["matches"])


def LO_hyp(**kw):
    import yolo_oracle as O

    h = O.scaled_hyp()
    h.update(kw)
    return h


def test_shared_cells_sum_gradients_and_last_match_wins():
    """Several matches on one cell: box and class gradients sum over them, tobj is the last in the reference's order."""
    p, t, anchors, hyp = loss_edge_inputs(FAMILIES["shared_cells"], 5)
    r = _compare(p, t, anchors, hyp)
    counts = {}
    for l, m in enumerate(r["matches"]):
        for cell in zip(m["b"].tolist(), m["a"].tolist(), m["gj"].tolist(), m["gi"].tolist()):
            counts[(l,) + cell] = counts.get((l,) + cell, 0) + 1
    assert max(counts.values()) >= 3
    # distinct classes on one cell (the class gradient of both is present)
    classes = {}
    for l, m in enumerate(r["matches"]):
        for k, cell in enumerate(zip(m["b"].tolist(), m["a"].tolist(), m["gj"].tolist(), m["gi"].tolist())):
            classes.setdefault((l,) + cell, set()).add(int(m["cls"][k]))
    assert max(len(c) for c in classes.values()) >= 2


def test_no_targets():
    anchors = grid_anchors("yolov3")
    g = torch.Generator().manual_seed(3)
    p = [torch.randn(2, 3, n, n, 85, generator=g) for n in (40, 20, 10)]
    r = _compare(p, torch.zeros(0, 6), anchors, LO_hyp())
    assert r["items"][0] == 0 and r["items"][2] == 0


def test_upstream_gradient_and_no_grad():
    p, t, anchors, hyp = loss_edge_inputs(_spec(), 61)
    r = LO.compute_loss(p, t, anchors, hyp)
    loss, items, grads = _kernel(p, t, anchors, hyp, upstream=2.5)
    for g, ref in zip(grads, r["grads"]):
        ref = 2.5 * ref
        assert np.all(np.abs(g - ref) <= 1e-4 * np.abs(ref) + 1e-6 * np.abs(ref).max())
    pc = [x.cuda() for x in p]  # inputs without requires_grad: same loss, nothing to differentiate
    l2, i2 = _loss(anchors, 80, hyp)(pc, t.cuda())
    assert not l2.requires_grad
    # equal up to the order of the kernel's double-precision atomic sums
    assert np.isclose(float(l2), loss, rtol=1e-6, atol=0) and np.allclose(i2.cpu().numpy(), items, rtol=1e-6, atol=0)


def test_malformed_rows_are_dropped():
    """Label rows with an image index outside [0, bs) or a class outside [0, nc) are ignored by the kernel: they match
    nothing and do not count in the means.  (The reference indexes with them: it raises on b >= bs or cls >= nc and wraps
    negative values.  Neither kind of row comes out of the reference's dataloader.)  The kernel on all rows must equal the
    restatement on the valid rows."""
    p, t, anchors, hyp = loss_edge_inputs(_spec(bs=2, nc=5), 62)
    bad = t[:4].clone()
    bad[0, 0], bad[1, 0], bad[2, 1], bad[3, 1] = 2.0, -1.0, 5.0, -1.0
    mixed = torch.cat((t[:3], bad[:2], t[3:], bad[2:]))
    _compare(p, mixed, anchors, hyp, t_ref=t)


def test_scale_bs16_and_crowd():
    """bs 16 at 640 with about 50 targets per image, plus one crowd image of 300 targets (many shared cells)."""
    import yolo_oracle as O

    g = torch.Generator().manual_seed(64)
    t = O.synth_targets(16, seed=64)
    rows = [t]
    for b in range(16):  # top up to ~50 per image
        n = 50 - int((t[:, 0] == b).sum())
        xy = torch.rand(n, 2, generator=g) * 0.9 + 0.05
        wh = torch.rand(n, 2, generator=g) * 0.3 + 0.01
        rows.append(torch.cat((torch.full((n, 1), float(b)), torch.randint(0, 80, (n, 1), generator=g).float(), xy, wh), 1))
    xy = torch.rand(300, 2, generator=g) * 0.4 + 0.3  # the crowd: 300 targets in the middle of image 5
    wh = torch.rand(300, 2, generator=g) * 0.1 + 0.02
    rows.append(torch.cat((torch.full((300, 1), 5.0), torch.randint(0, 80, (300, 1), generator=g).float(), xy, wh), 1))
    t = torch.cat(rows)
    p = [torch.randn(16, 3, n, n, 85, generator=g) for n in (80, 40, 20)]
    _compare(p, t, grid_anchors("yolov3"), LO_hyp())


@pytest.mark.parametrize("nl,na", [(6, 3), (3, 7)])
def test_beyond_abi_maxima_raises(nl, na):
    anchors = torch.ones(nl, na, 2)
    with pytest.raises(ValueError):
        _loss(anchors, 80, LO_hyp())


def test_abi_rejects_beyond_maxima():
    """The C ABI refuses nl > Y3_MAX_LEVELS / na > Y3_MAX_ANCHORS itself, whatever the caller."""
    import ctypes as C

    from yolov3_b200 import _lib

    L = _lib.lib()
    ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    out = torch.empty(4, device="cuda")
    for nl, na in ((6, 3), (3, 7)):
        d = _lib.LossDesc()
        d.nl, d.bs, d.na, d.nc, d.nt = nl, 1, na, 80, 0
        if nl == 6:
            assert L.y3_loss_workspace_bytes(C.byref(d)) < 0
        assert L.y3_loss_fwd_bwd(C.byref(d), ws.data_ptr(), ws.numel(), out.data_ptr(), None) != 0


@pytest.mark.parametrize("name", list(EDGE))
def test_loss_edge_golden(name):
    """Every reference golden of loss_edge_cases.npz through the kernel, at the tolerances of test_loss_golden."""
    g = np.load(G / "loss_edge_cases.npz")
    p, t, anchors, hyp = loss_edge_inputs(EDGE[name], int(g[f"{name}/seed"]))
    assert np.array_equal(t.numpy(), g[f"{name}/targets"]) and hyp == ast.literal_eval(str(g[f"{name}/hyp"]))
    loss, items, grads = _kernel(p, t, anchors, hyp)
    assert np.allclose(loss, g[f"{name}/loss"], rtol=1e-5)
    assert np.allclose(items, g[f"{name}/items"], rtol=1e-5, atol=1e-7)
    for i, got in enumerate(grads):
        ref = g[f"{name}/grad{i}"]
        assert np.allclose(got, ref, rtol=1e-4, atol=2e-7), (name, i, np.abs(got - ref).max())


"""Generate tests/golden/metrics_cases.npz by running the REFERENCE ITSELF (a checkout of ultralytics/yolov3 @ 97b87b1,
imported unmodified through oracle/ref_shim.py): utils/metrics.py's ap_per_class and ConfusionMatrix.process_batch on seeded
inputs, and val.py:424-428's summary numbers on the val images pinned in seam_cases.npz.  Before anything is written, the
CPU restatement in tests/metrics_oracle.py must agree with the reference on every case.

    python tests/golden/make_metrics_golden.py --reference <checkout>

Keys:
  ap/<case>/{tp,conf,pred_cls,target_cls}   inputs (bool [n, niou], float32 [n], float32 [n], float32 [nt])
  ap/<case>/{out_tp,out_fp,p,r,f1,ap,cls}   the reference's returned tuple
  ap/<case>/i                               the F1 index (the oracle's, once its p / r / f1 equal the reference's there)
  cm/<case>/{det,counts,labels,nc}          a sequence of images as one padded batch: det [bs, max_det, 6] + counts [bs],
                                            labels [nl, 6] = (image, cls, xyxy); count -1 = the detections=None call
  cm/<case>/matrix                          ConfusionMatrix(nc).matrix after process_batch on every image in order
  seam/{any,mp,mr,map50,map,ap50,ap,cls,nt,p,r,tp,fp}
                                            val.py:424-429 on the stats of seam_cases.npz's val images (nc = 80)
The large cases are generated from seeds inside the tests; this file stays small.
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT / "oracle"))
sys.path.insert(0, str(ROOT / "tests"))
import metrics_oracle as MO  # noqa: E402
import ref_shim  # noqa: E402
import yolo_oracle as O  # noqa: E402

OUT = Path(__file__).resolve().parent / "metrics_cases.npz"


def ap_case_list():
    """(name, kwargs of metrics_oracle.synth_stats, edit) — no confidence ties (the reference's order is unspecified there)."""
    def label_no_pred(tp, conf, pc, tc):
        tc = np.concatenate((tc, np.full(7, 11, np.float32)))  # class 11 has labels, no prediction carries it
        return tp, conf, pc, tc

    def pred_no_label(tp, conf, pc, tc):
        pc = pc.copy()
        pc[::9] = 12.0  # class 12 is predicted but has no labels
        return tp & (pc != 12.0)[:, None], conf, pc, tc

    return [
        ("typical", dict(n=3000, nc=10, n_targets=500, seed=0), None),
        ("crowded", dict(n=6000, nc=3, n_targets=900, seed=1, p_tp=0.5), None),
        ("sparse", dict(n=400, nc=40, n_targets=60, seed=2, p_tp=0.2), None),
        ("label_no_pred", dict(n=800, nc=8, n_targets=120, seed=3), label_no_pred),
        ("pred_no_label", dict(n=800, nc=8, n_targets=120, seed=4), pred_no_label),
        ("one_row", dict(n=1, nc=1, n_targets=1, seed=5, p_tp=3.0), None),
        ("niou1", dict(n=1500, nc=6, n_targets=250, niou=1, seed=6), None),
    ]


def gen_ap(store):
    from utils.metrics import ap_per_class  # reference

    for name, kw, edit in ap_case_list():
        tp, conf, pc, tc = MO.synth_stats(**kw)
        if edit:
            tp, conf, pc, tc = edit(tp, conf, pc, tc)
        ref = ap_per_class(tp.copy(), conf.copy(), pc.copy(), tc.copy(), plot=False, names={})
        ora = MO.ap_per_class(tp, conf, pc, tc)
        o = ora["ref"]
        assert np.array_equal(ref[5], o[5]), (name, "ap", np.abs(ref[5] - o[5]).max())  # bit-exact AP
        for k in (2, 3, 4):
            assert np.allclose(ref[k], o[k], rtol=0, atol=1e-12), (name, k)
        for k in (0, 1, 6):
            assert np.array_equal(ref[k], o[k]), (name, k)
        assert ref[0].dtype == np.float64 and ref[6].dtype == o[6].dtype
        for k, v in (("tp", tp), ("conf", conf), ("pred_cls", pc), ("target_cls", tc)):
            store[f"ap/{name}/{k}"] = v
        for k, v in zip(("out_tp", "out_fp", "p", "r", "f1", "ap", "cls"), ref):
            store[f"ap/{name}/{k}"] = v
        store[f"ap/{name}/i"] = np.array(ora["i"])
        print("ap", name, tp.shape, "classes", len(ref[6]), "mAP50", float(ref[5][:, 0].mean()) if len(ref[6]) else None)


def cm_case_list():
    """(name, nc, images): image = (det [N, 6] or None, labels [M, 5] = (cls, xyxy))."""
    out = []
    imgs = []
    for i, (nd, nl, seed, jit) in enumerate([(60, 12, 0, 8.0), (0, 5, 1, 1.0), (25, 6, 2, 6.0), (120, 30, 3, 4.0)]):
        d, l = O.synth_val_case(nd, nl, 5, seed=30 + seed, jitter=jit)
        imgs.append((d if nd else None, l))
    d, l = O.synth_val_case(20, 4, 5, seed=40)
    d[:, 4] = d[:, 4] * 0.2  # every detection under conf 0.25
    imgs.append((d, l))
    d, l = O.synth_val_case(15, 4, 5, seed=41)
    d[:, :4] = torch.tensor([600.0, 600.0, 630.0, 630.0]) + torch.arange(15.0)[:, None] * 0.01
    d[:, 4] = 0.9  # detections kept but far from every label: no match, so unmatched detections are not counted
    l[:, 1:] = l[:, 1:].clamp(max=500.0)
    imgs.append((d, l))
    d, l = O.synth_val_case(200, 40, 3, seed=42, jitter=2.0)  # dense overlaps
    imgs.append((d, l))
    out.append(("sequence", 5, imgs))
    out.append(("dense", 3, [O.synth_val_case(300, 60, 3, seed=50 + k, jitter=3.0) for k in range(3)]))
    return out


def pad_batch(imgs):
    bs = len(imgs)
    max_det = max([1] + [len(d) for d, _ in imgs if d is not None])
    det = np.zeros((bs, max_det, 6), np.float32)
    counts = np.zeros(bs, np.int32)
    labels = []
    for i, (d, l) in enumerate(imgs):
        if d is None:
            counts[i] = -1
        else:
            det[i, : len(d)] = d.numpy()
            counts[i] = len(d)
        labels.append(np.concatenate((np.full((len(l), 1), i, np.float32), l.numpy()), 1))
    return det, counts, np.concatenate(labels, 0)


def gen_cm(store):
    from utils.metrics import ConfusionMatrix  # reference

    for name, nc, imgs in cm_case_list():
        cm = ConfusionMatrix(nc=nc)
        ora = np.zeros((nc + 1, nc + 1), np.int64)
        for d, l in imgs:
            if d is None:
                cm.process_batch(detections=None, labels=l[:, 0])
                MO.confusion_update(ora, None, l[:, 0].numpy(), nc)
            else:
                cm.process_batch(d, l)
                MO.confusion_update(ora, d.numpy(), l.numpy(), nc)
        assert np.array_equal(cm.matrix, ora), (name, cm.matrix, ora)
        det, counts, labels = pad_batch(imgs)
        store[f"cm/{name}/det"], store[f"cm/{name}/counts"], store[f"cm/{name}/labels"] = det, counts, labels
        store[f"cm/{name}/nc"], store[f"cm/{name}/matrix"] = np.array(nc), cm.matrix
        print("cm", name, "images", len(imgs), "total", int(cm.matrix.sum()))


def gen_seam(store):
    from utils.metrics import ap_per_class  # reference

    g = np.load(OUT.parent / "seam_cases.npz")
    stats = []
    for si in range(2):
        out, labelsn, correct = g[f"val/{si}/out"], g[f"val/{si}/labelsn"], g[f"val/{si}/correct"]
        stats.append((correct, out[:, 4], out[:, 5], labelsn[:, 0]))
    stats = [np.concatenate(x, 0) for x in zip(*stats)]  # val.py:424
    # val.py:425 calls ap_per_class only when some detection is a true positive; these synthetic predictions have none, so
    # the summary is val.py's zeros.  The per-class numbers of the ungated call are pinned as well.
    gate = bool(stats[0].any())
    tp, fp, p, r, f1, ap, ap_class = ap_per_class(*stats, plot=False, names={})
    ora = MO.ap_per_class(*stats, nc=80)["ref"]
    assert np.array_equal(ap, ora[5]) and np.array_equal(ap_class, ora[6])
    assert np.array_equal(p, ora[2]) and np.array_equal(r, ora[3]) and np.array_equal(tp, ora[0]) and np.array_equal(fp, ora[1])
    ap50, ap = ap[:, 0], ap.mean(1)  # val.py:427-428
    mp, mr, map50, map_ = (p.mean(), r.mean(), ap50.mean(), ap.mean()) if gate else (0.0, 0.0, 0.0, 0.0)
    nt = np.bincount(stats[3].astype(int), minlength=80)  # val.py:429
    for k, v in (("any", gate), ("mp", mp), ("mr", mr), ("map50", map50), ("map", map_), ("ap50", ap50), ("ap", ap),
                 ("cls", ap_class), ("nt", nt), ("p", p), ("r", r), ("tp", tp), ("fp", fp)):
        store[f"seam/{k}"] = np.asarray(v)
    print("seam", dict(any=gate, mp=mp, mr=mr, map50=map50, map=map_), "classes", len(ap_class), "rows", len(stats[1]))


if __name__ == "__main__":
    args = sys.argv[1:]
    if "--reference" in args:
        i = args.index("--reference")
        ref_shim.REFERENCE_ROOT = Path(args[i + 1]).resolve()
        del args[i:i + 2]
    assert ref_shim.reference_available(), "pass --reference <checkout of ultralytics/yolov3 @ 97b87b1>"
    ref_shim.install()
    torch.set_num_threads(8)
    store = {}
    gen_ap(store)
    gen_cm(store)
    gen_seam(store)
    np.savez_compressed(OUT, **store)
    print("wrote", OUT, OUT.stat().st_size, "bytes")

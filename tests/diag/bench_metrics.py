"""Device vs host time of the validation metrics at COCO-val size, on identical inputs, with an output check.

    python tests/diag/bench_metrics.py [--out profiles/r03_metrics.json] [--iters 20] [--host-images 5000]

  device: ap_per_class_batched on 5000 images x 300 padded rows x 10 IoU thresholds, 80 classes, and
          ConfusionMatrix.process_batch_batched over 5000 images in batches of 32; CUDA events around the calls, after warm-up.
          ap_per_class reads ~52 MB of padded rows (det 36 MB, correct 15 MB, labels) and sorts in ~42 MB of workspace, about
          94 MB in all: below the B200's 126 MB L2, so successive timed calls are partly served from L2 (the cache is not
          flushed between calls).  The matrix pass reads 36 MB of detections per pass.
  host:   the reference's own ap_per_class and per-image ConfusionMatrix (utils/metrics.py) from the copy build() stages under
          oracle/_ref, through oracle/ref_shim.py; where that copy is absent, the CPU restatement in tests/metrics_oracle.py,
          labelled as such.  Timed once (they take seconds).
The card name and power limit are read in the same run and written next to the numbers."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))
sys.path.insert(0, str(ROOT / "tests"))
import metrics_oracle as MO  # noqa: E402
from test_metrics_gpu import _cm_images, _coco_sized  # noqa: E402  (the same seeded inputs as the full-scale tests)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = (s.strip() for s in q.split(","))
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def time_device(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)), "iters": iters}


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", default=None)
    ap_.add_argument("--iters", type=int, default=20)
    ap_.add_argument("--host-images", type=int, default=5000, help="images the host ConfusionMatrix loop runs over")
    args = ap_.parse_args()
    assert torch.cuda.is_available(), "bench_metrics.py measures the device: it needs a CUDA GPU"
    from yolov3_b200.metrics import ConfusionMatrix, ap_per_class_batched

    import ref_shim

    use_ref = ref_shim.reference_available()
    if use_ref:
        ref_shim.install()
        from utils.metrics import ConfusionMatrix as HostCM  # reference
        from utils.metrics import ap_per_class as host_ap  # reference
        host_label = "reference utils/metrics.py (staged copy under oracle/_ref)"
    else:
        host_label = "CPU restatement tests/metrics_oracle.py (the staged reference copy is absent)"
    result = {"card": card(), "host": {"implementation": host_label, "cpu_count": os.cpu_count(),
                                       "torch_threads": torch.get_num_threads()}}

    # ---- ap_per_class
    det, counts, correct, labels, (tp, conf, pc, tc) = _coco_sized()
    d = [torch.from_numpy(x).cuda() for x in (det, counts, correct, labels)]
    dev = time_device(lambda: ap_per_class_batched(d[0], d[1], d[2], d[3], 80), args.iters)
    res = {k: v.cpu().numpy() for k, v in ap_per_class_batched(*d, 80)._asdict().items()}
    t0 = time.perf_counter()
    if use_ref:
        h = host_ap(tp, conf, pc, tc, plot=False, names={})
    else:
        h = MO.ap_per_class(tp, conf, pc, tc, nc=80)["ref"]
    host_s = time.perf_counter() - t0
    cls = np.flatnonzero(res["present"])
    match = {"ap_bit_identical": bool(np.array_equal(res["ap"][cls], h[5])),
             "p_r_f1_max_abs_diff": float(max(np.abs(res[k][cls] - h[i]).max() for k, i in (("p", 2), ("r", 3), ("f1", 4)))),
             "tp_fp_classes_equal": bool(np.array_equal(res["tp"][cls], h[0]) and np.array_equal(res["fp"][cls], h[1])
                                         and np.array_equal(cls, h[6]))}
    result["ap_per_class"] = {"shape": {"images": 5000, "rows_per_image": 300, "valid_rows": int(counts.sum()), "niou": 10,
                                        "nc": 80, "labels": len(tc)},
                              "device": dev, "host_s": host_s, "outputs": match}
    print("ap_per_class", json.dumps(result["ap_per_class"]), flush=True)

    # ---- ConfusionMatrix
    cdet, ccounts, clabels = _cm_images(3)
    nimg, bs = len(ccounts), 32
    batches = []
    for b0 in range(0, nimg, bs):
        sel = (clabels[:, 0] >= b0) & (clabels[:, 0] < b0 + bs)
        lab = clabels[sel].copy()
        lab[:, 0] -= b0
        batches.append((torch.from_numpy(cdet[b0:b0 + bs]).cuda(), torch.from_numpy(ccounts[b0:b0 + bs]).cuda(),
                        torch.from_numpy(lab).cuda()))

    def run_cm():
        cm = ConfusionMatrix(80)
        for x in batches:
            cm.process_batch_batched(*x)
        return cm

    cdev = time_device(run_cm, max(3, args.iters // 4))
    got = run_cm().matrix
    nh = min(args.host_images, nimg)
    host_m = np.zeros((81, 81))
    t0 = time.perf_counter()
    if use_ref:
        hc = HostCM(nc=80)
        for i in range(nh):
            lab = torch.from_numpy(clabels[clabels[:, 0] == i, 1:])
            if len(lab) == 0:
                continue
            if ccounts[i] == 0:
                hc.process_batch(detections=None, labels=lab[:, 0])
            else:
                hc.process_batch(torch.from_numpy(cdet[i, : ccounts[i]]), lab)
        host_m = hc.matrix
    else:
        mo = np.zeros((81, 81), np.int64)
        for i in range(nh):
            lab = clabels[clabels[:, 0] == i, 1:]
            if len(lab):
                MO.confusion_update(mo, None if ccounts[i] == 0 else cdet[i, : ccounts[i]],
                                    lab[:, 0] if ccounts[i] == 0 else lab, 80)
        host_m = mo.astype(np.float64)
    host_cm_s = time.perf_counter() - t0
    result["confusion_matrix"] = {"shape": {"images": nimg, "batch": bs, "max_det": 300, "labels": len(clabels), "nc": 80},
                                  "device": cdev, "host_s": host_cm_s, "host_images": nh,
                                  "outputs": {"matrix_equal": bool(nh == nimg and np.array_equal(got, host_m))}}
    print("confusion_matrix", json.dumps(result["confusion_matrix"]), flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    ok = match["ap_bit_identical"] and match["tp_fp_classes_equal"] and match["p_r_f1_max_abs_diff"] <= 1e-12
    ok = ok and result["confusion_matrix"]["outputs"]["matrix_equal"]
    print(json.dumps(result))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()

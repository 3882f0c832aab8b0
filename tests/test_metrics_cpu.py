"""The CPU restatement of the validation metrics (tests/metrics_oracle.py) against the goldens recorded from the reference's
own ap_per_class / ConfusionMatrix (tests/golden/make_metrics_golden.py), and its interp / trapezoid pieces against numpy."""
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
import metrics_oracle as MO  # noqa: E402

G = Path(__file__).parent / "golden" / "metrics_cases.npz"


def _cases(prefix):
    g = np.load(G)
    return sorted({k.split("/")[1] for k in g.files if k.startswith(prefix + "/")})


@pytest.mark.parametrize("case", _cases("ap"))
def test_oracle_ap_per_class_matches_reference_golden(case):
    g = np.load(G)
    k = f"ap/{case}/"
    o = MO.ap_per_class(g[k + "tp"], g[k + "conf"], g[k + "pred_cls"], g[k + "target_cls"])
    tp, fp, p, r, f1, ap, cls = o["ref"]
    assert np.array_equal(ap, g[k + "ap"])  # bit-exact
    for got, key in ((p, "p"), (r, "r"), (f1, "f1")):
        assert np.allclose(got, g[k + key], rtol=0, atol=1e-12), key
    assert np.array_equal(tp, g[k + "out_tp"]) and np.array_equal(fp, g[k + "out_fp"])
    assert np.array_equal(cls, g[k + "cls"])
    assert o["i"] == int(g[k + "i"])


@pytest.mark.parametrize("case", _cases("cm"))
def test_oracle_confusion_matrix_matches_reference_golden(case):
    g = np.load(G)
    k = f"cm/{case}/"
    nc, det, counts, labels = int(g[k + "nc"]), g[k + "det"], g[k + "counts"], g[k + "labels"]
    m = np.zeros((nc + 1, nc + 1), np.int64)
    for i in range(len(counts)):
        lab = labels[labels[:, 0] == i, 1:]
        if counts[i] < 0:
            MO.confusion_update(m, None, lab[:, 0], nc)
        else:
            MO.confusion_update(m, det[i, : counts[i]], lab, nc)
    assert np.array_equal(m, g[k + "matrix"])


def test_oracle_seam_summary_matches_reference_golden():
    g = np.load(G)
    s = np.load(Path(__file__).parent / "golden" / "seam_cases.npz")
    stats = [np.concatenate(x, 0) for x in zip(*[(s[f"val/{si}/correct"], s[f"val/{si}/out"][:, 4], s[f"val/{si}/out"][:, 5],
                                                  s[f"val/{si}/labelsn"][:, 0]) for si in range(2)])]
    o = MO.ap_per_class(*stats, nc=80)
    tp, fp, p, r, f1, ap, cls = o["ref"]
    assert bool(stats[0].any()) == bool(g["seam/any"])
    assert np.array_equal(ap[:, 0], g["seam/ap50"]) and np.array_equal(ap.mean(1), g["seam/ap"])
    assert np.array_equal(cls, g["seam/cls"]) and np.array_equal(o["nt"], g["seam/nt"])
    assert np.array_equal(p, g["seam/p"]) and np.array_equal(r, g["seam/r"])


def _monotone(rng, n, dup):
    x = np.sort(rng.random(n))
    if dup:
        x[rng.integers(1, n, n // 4)] = x[rng.integers(0, n, n // 4)]
        x = np.sort(x)
    return x


@pytest.mark.parametrize("seed", range(4))
def test_interp_and_trapezoid_restatements_are_numpy_bit_for_bit(seed):
    rng = np.random.default_rng(seed)
    for trial in range(60):
        n = int(rng.integers(1, 300))
        xp = _monotone(rng, n, dup=trial % 2 == 1)
        if trial % 3 == 0:
            xp = np.concatenate(([0.0], xp, [1.0]))
        fp = rng.random(len(xp))
        x = np.concatenate((MO.AP_X, rng.random(50) * 1.2 - 0.1, xp[: min(len(xp), 10)]))
        for left in (None, 0.0, 1.0):
            assert np.array_equal(MO.interp(x, xp, fp, left=left), np.interp(x, xp, fp, left=left)), (trial, left)
        y = rng.random(101)
        assert MO.trapezoid(y, MO.AP_X) == np.trapezoid(y, np.linspace(0, 1, 101))
    assert np.array_equal(MO.AP_X, np.linspace(0, 1, 101)) and np.array_equal(MO.PX, np.linspace(0, 1, 1000))


@pytest.mark.parametrize("seed", range(3))
def test_compute_ap_restatement_is_the_reference_formula_bit_for_bit(seed):
    """compute_ap as the reference writes it (np.maximum.accumulate envelope, np.interp, np.trapezoid) vs the restatement."""
    rng = np.random.default_rng(100 + seed)
    for _ in range(100):
        n_l, m = int(rng.integers(1, 40)), int(rng.integers(1, 200))
        t = (rng.random(m) < 0.3).astype(np.int64)
        t[np.cumsum(t) > n_l] = 0
        tpc, fpc = np.cumsum(t), np.cumsum(1 - t)
        recall, precision = tpc / (n_l + 1e-16), tpc / (tpc + fpc)
        mrec = np.concatenate(([0.0], recall, [1.0]))
        mpre = np.flip(np.maximum.accumulate(np.flip(np.concatenate(([1.0], precision, [0.0])))))
        x = np.linspace(0, 1, 101)
        assert MO.compute_ap(recall, precision) == np.trapezoid(np.interp(x, mrec, mpre), x)

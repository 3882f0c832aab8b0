"""The float64 restatement of ComputeLoss (tests/loss_oracle.py) against the goldens recorded from the reference's own
ComputeLoss (tests/golden/loss_cases.npz, loss_edge_cases.npz) and against the float32 oracle on the synthetic workload.
build_targets must agree exactly (indices, classes, anchors; tbox to fp32 rounding); the loss to 1e-5 and dL/dp to
1e-4 relative, which is the float32 reference's own error against the float64 restatement."""
import ast
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent))
sys.path.insert(0, str(Path(__file__).resolve().parent / "golden"))
import loss_oracle as LO  # noqa: E402
import yolo_oracle as O  # noqa: E402
from make_golden import loss_edge_case_list, loss_edge_inputs, loss_inputs  # noqa: E402

G = Path(__file__).parent / "golden"
EDGE = dict(loss_edge_case_list())


def _bt_table(m):
    return np.concatenate([np.stack([m[k] for k in ("b", "a", "gj", "gi")], 1), m["tbox"], m["anch"], m["cls"][:, None]], 1)


def _check(r, g, key, nl):
    assert np.allclose(r["loss"], g[f"{key}/loss"], rtol=1e-5, atol=0)
    assert np.allclose(r["items"], g[f"{key}/items"], rtol=1e-5, atol=1e-7)
    for i in range(nl):
        ref = g[f"{key}/grad{i}"]
        assert np.allclose(r["grads"][i], ref, rtol=1e-4, atol=1e-6 * np.abs(ref).max()), (key, i)
        bt, got = g[f"{key}/bt{i}"], _bt_table(r["matches"][i])
        assert got.shape == bt.shape, (key, i)
        assert np.array_equal(got[:, :4], bt[:, :4]) and np.array_equal(got[:, 8:], bt[:, 8:]), (key, i)  # b a gj gi, cls
        assert np.array_equal(got[:, 6:8], bt[:, 6:8])  # anchors
        assert np.allclose(got[:, 4:6], bt[:, 4:6], rtol=0, atol=1e-6)  # tbox xy: fp32 gxy - gij


@pytest.mark.parametrize("case", range(4))
def test_restatement_matches_loss_golden(case):
    g = np.load(G / "loss_cases.npz")
    hyp = ast.literal_eval(str(g["hyp"]))
    p, t = loss_inputs(case)
    r = LO.compute_loss(p, t, torch.from_numpy(g["anchors"]), hyp)
    _check(r, g, f"c{case}", 3)


@pytest.mark.parametrize("name", list(EDGE))
def test_restatement_matches_loss_edge_golden(name):
    g = np.load(G / "loss_edge_cases.npz")
    p, t, anchors, hyp = loss_edge_inputs(EDGE[name], int(g[f"{name}/seed"]))
    assert np.array_equal(t.numpy(), g[f"{name}/targets"])
    assert hyp == ast.literal_eval(str(g[f"{name}/hyp"]))
    r = LO.compute_loss(p, t, anchors, hyp)
    _check(r, g, name, len(p))


def test_edge_golden_covers_the_index_clamp():
    """The image-edge case has centres at x or y = 1.0: the clamped cell nx - 1 (ny - 1) gets tbox x (y) = 1.0, which is what
    the reference computes (its gi, gj are views of gij, clamped in place before tbox is formed)."""
    g = np.load(G / "loss_edge_cases.npz")
    for i in range(3):
        bt = g[f"image_edge/bt{i}"]
        assert (bt[:, 4] == 1.0).any() and (bt[:, 5] == 1.0).any(), i
        assert bt[:, 4].max() <= 1.5 and bt[:, 5].max() <= 1.5


def test_restatement_matches_oracle_on_synth_targets():
    anchors = O.init_params(Path(__file__).resolve().parents[1] / "yolov3_b200" / "cfg" / "yolov3.yaml")["model.28.anchors"]
    hyp = O.scaled_hyp()
    g = torch.Generator().manual_seed(4)
    p = [torch.randn(3, 3, s, s, 85, generator=g) for s in (32, 16, 8)]
    t = O.synth_targets(3, seed=11)
    po = [x.clone().requires_grad_(True) for x in p]
    lo, io = O.compute_loss(po, t, anchors, hyp)
    lo.backward()
    r = LO.compute_loss(p, t, anchors, hyp)
    assert np.allclose(r["loss"], float(lo.detach()), rtol=1e-5)
    assert np.allclose(r["items"], io.numpy(), rtol=1e-5, atol=1e-7)
    for a, b in zip(r["grads"], po):
        ref = b.grad.numpy()
        assert np.allclose(a, ref, rtol=1e-4, atol=1e-6 * np.abs(ref).max())
    bt = O.build_targets([tuple(x.shape) for x in p], t, anchors, hyp["anchor_t"])
    for i in range(3):
        for k in ("b", "a", "gj", "gi"):
            assert np.array_equal(r["matches"][i][k], bt[i][k].numpy()), (i, k)
        assert np.array_equal(r["matches"][i]["cls"], bt[i]["tcls"].numpy())
        assert np.allclose(r["matches"][i]["tbox"], bt[i]["tbox"].numpy(), rtol=0, atol=1e-6)

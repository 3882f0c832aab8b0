"""Host logic of the training path that needs no GPU: the flat parameter store (``params.ParamStore``) — reference parameter
names / shapes, aliasing views with the conv kernel's K-major order, optimizer groups as utils/torch_utils.py:207-237
(smart_optimizer) forms them, and the all-reduce bucket partition of the gradient buffer (utils/torch_utils.py:60-72 gets its
overlap from DDP's buckets)."""
from pathlib import Path

import pytest
import torch

import yolo_oracle as O

ROOT = Path(__file__).resolve().parents[1]
CFG = ROOT / "yolov3_b200" / "cfg"


def _store(name):
    from yolov3_b200 import params as P
    from yolov3_b200.model import Model

    m = Model(CFG / f"{name}.yaml", device="cpu")
    m.load_state_dict(O.init_params(CFG / f"{name}.yaml", seed=0))
    return m, m.store(), P


@pytest.mark.parametrize("name", ["yolov3", "yolov3-spp", "yolov3-tiny"])
def test_flat_store_layout_and_groups(name):
    m, st, P = _store(name)
    ref = O.init_params(CFG / f"{name}.yaml", seed=0)
    # every reference-named tensor is a view of ONE flat buffer, with the reference's logical shape and values
    assert list(st.views) == list(ref)
    base = st.P.untyped_storage().data_ptr()
    for k, v in st.views.items():
        assert tuple(v.shape) == tuple(ref[k].shape), k
        assert v.untyped_storage().data_ptr() == base, k
        assert torch.equal(v.detach(), ref[k]), k
    # slots: 256-element aligned, disjoint, trainables first (backward-completion order: heads, then blocks last-to-first)
    off = 0
    for nm in st.order:
        s = st.slots[nm]
        assert s.offset == off and s.numel % P.CHUNK == 0 and s.numel >= int(torch.tensor(s.shape).prod())
        off += s.numel
    assert off == st.n_total and st.n_train < st.n_total and st.G.numel() == st.n_train
    train_names = [n for n in st.order if st.slots[n].group != P.G_FROZEN]
    assert [st.slots[n].offset for n in train_names] == sorted(st.slots[n].offset for n in train_names)
    assert st.slots[train_names[-1]].offset + st.slots[train_names[-1]].numel == st.n_train
    det = m.detect.i
    assert train_names[0] == f"model.{det}.m.0.weight" and train_names[-1].startswith("model.0.")
    conv_idx = [int(n.split(".")[1]) for n in train_names if n.endswith("conv.weight")]
    assert conv_idx == sorted(conv_idx, reverse=True)
    # a conv weight's storage order is [co][kh][kw][ci] (channels_last strides of [co,ci,k,k]): the forward pack is a VIEW
    w = next(n for n in train_names if n.endswith("conv.weight") and st.slots[n].taps == 9)
    s = st.slots[w]
    co, ci, k, _ = s.shape
    assert s.stride == (k * k * ci, 1, k * ci, ci)
    packed = st.P[s.offset:s.offset + co * 9 * ci].view(co, 3, 3, ci)
    assert torch.equal(packed, ref[w].permute(0, 2, 3, 1))
    # optimizer groups exactly as smart_optimizer forms them: bias -> g2, BatchNorm weight -> g1, everything else -> g0 (decay)
    groups = {0: [], 1: [], 2: []}
    for n in train_names:
        groups[st.slots[n].group].append(n)
    assert all(n.endswith("bias") for n in groups[P.G_BIAS]) and all(n.endswith("bn.weight") for n in groups[P.G_BN])
    assert all(n.endswith("conv.weight") or (f"model.{det}.m." in n and n.endswith(".weight")) for n in groups[P.G_DECAY])
    n_conv = sum(1 for k in ref if k.endswith("conv.weight"))
    nl = m.detect.nl
    assert (len(groups[0]), len(groups[1]), len(groups[2])) == (n_conv + nl, n_conv, n_conv + nl)
    # the per-256-element group map the fused SGD kernel reads agrees with the slots; buffers are frozen
    gm = st.group.cpu()
    for n in st.order:
        s = st.slots[n]
        assert bool((gm[s.offset // P.CHUNK:(s.offset + s.numel) // P.CHUNK] == s.group).all()), n
    assert all(st.slots[n].group == P.G_FROZEN for n in st.order if "running_" in n or n.endswith("anchors"))
    # gradient views alias the flat gradient buffer with the parameter's strides; attach / detach keeps them in place
    st.attach_grads()
    gb = st.G.untyped_storage().data_ptr()
    for n in train_names:
        p = st.views[n]
        assert p.requires_grad and p.grad is st.grads[n] and p.grad.untyped_storage().data_ptr() == gb
        assert p.grad.stride() == p.stride() and p.grad.storage_offset() == p.storage_offset()
    assert st.grads_are_live()
    st.zero_grad(set_to_none=True)
    assert not st.grads_are_live() and all(st.views[n].grad is None for n in train_names)


def test_reference_smart_optimizer_groups_agree():
    """The same three groups as the REFERENCE's smart_optimizer forms (tests/golden/seam_cases.npz: parameter names per
    group and each group's weight decay), on the nn.Module facade's parameters."""
    import numpy as np

    from yolov3_b200 import params as P
    from yolov3_b200.module import DetectionModel

    g = np.load(ROOT / "tests" / "golden" / "seam_cases.npz")
    dm = DetectionModel(CFG / "yolov3-tiny.yaml", device="cpu")
    st = dm.core.store()
    named = dict(dm.named_parameters())
    by_ptr = {st.views[n].data_ptr(): n for n in st.order if st.slots[n].group != P.G_FROZEN}
    got = {}
    for gi, tag in enumerate((P.G_BIAS, P.G_DECAY, P.G_BN)):  # smart_optimizer: g2 first, then g0 (decay), g1
        for name in g[f"optim/yolov3-tiny/{gi}/names"]:
            got[by_ptr[named[str(name)].data_ptr()]] = tag
        assert (g[f"optim/yolov3-tiny/{gi}/hyp"][3] > 0) == (tag == P.G_DECAY)
    assert got == {n: st.slots[n].group for n in by_ptr.values()}


@pytest.mark.parametrize("name,n_buckets", [("yolov3", 4), ("yolov3", 1), ("yolov3", 7), ("yolov3-tiny", 4)])
def test_gradient_bucket_partition(name, n_buckets):
    _, st, P = _store(name)
    r = st.bucket_ranges(n_buckets)
    assert 1 <= len(r) <= n_buckets and r[0][0] == 0 and r[-1][1] == st.n_train
    assert all(a[1] == b[0] for a, b in zip(r, r[1:])) and all(b > a for a, b in r)
    # slot-aligned: a parameter's gradient never straddles two buckets
    starts = {st.slots[n].offset for n in st.order}
    assert all(a in starts for a, _ in r)
    if n_buckets == 4 and name == "yolov3":
        sizes = [b - a for a, b in r]
        assert len(r) == 4 and sizes[-1] < 0.02 * st.n_train < min(sizes[:-1])  # the exposed tail bucket is the small one
        # ... and it holds the layers whose backward finishes last (model.0 ...)
        tail = [n for n in st.order if r[-1][0] <= st.slots[n].offset < r[-1][1]]
        assert any(n.startswith("model.0.") for n in tail) and all(int(n.split(".")[1]) <= 7 for n in tail)

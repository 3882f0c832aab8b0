"""Host-side logic that needs no GPU: the C-ABI library loads and exports every symbol include/yolov3_b200.h
declares, the ctypes mirrors match the C structs, the YAML lowering reproduces the reference graph contract, the
Python seams keep the reference's error behaviour, and the multi-rank aggregation works over gloo."""
import os
import re
import subprocess
import sys
from pathlib import Path

import pytest
import torch

import yolo_oracle as O

ROOT = Path(__file__).resolve().parents[1]
CFG = ROOT / "yolov3_b200" / "cfg"


def test_library_exports_every_declared_symbol():
    from yolov3_b200 import _lib

    L = _lib.lib()
    hdr = (ROOT / "include" / "yolov3_b200.h").read_text()
    names = set(re.findall(r"^\s*(?:int|int32_t|int64_t|void)\s+(y3_\w+)\s*\(", hdr, flags=re.M))
    assert len(names) >= 15
    for n in names:
        assert hasattr(L, n), f"{n} declared in the header but not exported"
    assert set(_lib.SYMBOLS) == names, (set(_lib.SYMBOLS) ^ names)
    assert L.y3_version() >= 100
    assert L.y3_conv_cout_pad(255) == 256 and L.y3_conv_cout_pad(32) == 32 and L.y3_conv_cout_pad(1024) == 1024
    assert L.y3_nms_default_capacity(25200, 80, 0) == 32768
    assert L.y3_nms_workspace_bytes(32, 32768) > 0


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from yolov3_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "_LIB_PATH", tmp_path / "nope.so")
    with pytest.raises(_lib.Y3Error, match="no CPU or PyTorch fallback"):
        _lib.lib()


@pytest.mark.parametrize("name", ["yolov3", "yolov3-spp", "yolov3-tiny"])
def test_graph_contract(name):
    from yolov3_b200 import graph
    from yolov3_b200.model import Model

    cfg, _ = graph.resolve_cfg(CFG / f"{name}.yaml")
    nodes, save = graph.parse(cfg)
    onodes, osave = O.parse_graph(CFG / f"{name}.yaml")
    assert save == osave
    assert [(n.type, n.n, n.c_out) for n in nodes] == [(n["type"], n["n"], n["c_out"]) for n in onodes]
    assert graph.strides(nodes) == O.detect_strides(onodes)
    assert [(c.prefix, c.c1, c.c2, c.k, c.s) for c in graph.conv_specs(nodes)] == O.conv_prefixes(onodes)
    m = Model(CFG / f"{name}.yaml", device="cpu")
    params = O.init_params(CFG / f"{name}.yaml", seed=0)
    assert list(m.state_dict().keys()) == list(params.keys())
    assert torch.allclose(m.detect.anchors, params[f"model.{m.detect.i}.anchors"])
    missing, unexpected = m.load_state_dict(params)
    assert not missing and not unexpected
    with pytest.raises(RuntimeError):
        m.load_state_dict({"bogus": torch.zeros(1)})
    n_params = sum(v.numel() for k, v in m.params.items() if "running" not in k and not k.endswith("anchors"))
    assert n_params == {"yolov3": 61949149, "yolov3-spp": 62998749, "yolov3-tiny": 8852366}[name]


def test_lowering_zero_copy_concat_and_fused_upsample():
    from yolov3_b200 import _lib
    from yolov3_b200.model import Engine, Model

    m = Model(CFG / "yolov3.yaml", device="cpu")
    e = Engine(m, 2, 64, 96, dry_run=True)
    kinds = [o.kind for o in e.op_list]
    assert kinds.count(_lib.OP_CONV) == 74 and kinds.count(_lib.OP_CONV_FIRST) == 1 and kinds[-1] == _lib.OP_DECODE
    convs = [o.conv for o in e.op_list if o.kind == _lib.OP_CONV]
    ups = [c for c in convs if c.upsample]
    assert [(c.c_in, c.c_out, c.out_ld, c.out_coff) for c in ups] == [(512, 256, 768, 0), (256, 128, 384, 0)]
    cat18 = e.bufs[18]
    # node 8's last bottleneck writes channels [256,768) of the node-18 buffer; node 9 reads them back from there
    w = [c for c in convs if c.out == cat18.ptr and not c.upsample]
    assert [(c.out_ld, c.out_coff, c.c_out) for c in w] == [(768, 256, 512)] and w[0].res
    r = [c for c in convs if c.in_ == cat18.ptr]
    assert sorted((c.in_coff, c.c_in, c.stride) for c in r) == [(0, 768, 1), (256, 512, 2)]
    heads = [c for c in convs if c.out_f32]
    assert [(c.c_in, c.c_out, c.act) for c in heads] == [(256, 255, 0), (512, 255, 0), (1024, 255, 0)]
    assert e.z.shape == (2, 3 * (8 * 12 + 4 * 6 + 2 * 3), 85)
    with pytest.raises(_lib.Y3Error):
        e.run(None)
    with pytest.raises(ValueError):
        Engine(m, 1, 100, 64, dry_run=True)  # not a multiple of the max stride


def test_reference_error_behaviour_at_the_seams():
    from yolov3_b200.model import Model
    from yolov3_b200.nms import non_max_suppression

    with pytest.raises(AssertionError):
        non_max_suppression(torch.zeros(1, 10, 85), conf_thres=1.2)
    with pytest.raises(AssertionError):
        non_max_suppression(torch.zeros(1, 10, 85), iou_thres=-1)
    with pytest.raises(AssertionError, match="no CPU path"):
        non_max_suppression(torch.zeros(1, 10, 85))
    m = Model(CFG / "yolov3-tiny.yaml", device="cpu")
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.zeros(1, 3, 64, 64))
    with pytest.raises(NotImplementedError):
        m(torch.zeros(1, 3, 64, 64), visualize=True)  # profile / visualize are outside the accelerated path; augment is built


WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from bench import aggregate
dist.init_process_group("gloo")
r = dist.get_rank()
ms = aggregate(100.0 + 50.0 * r, torch.device("cpu"))       # max over ranks
assert ms == 150.0, ms
if r == 0:
    print("AGG", ms, dist.get_world_size() * 32 * 10 / (ms / 1e3))
dist.barrier(); dist.destroy_process_group()
'''


def test_multi_rank_aggregation_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29653", str(script), str(ROOT)], capture_output=True, text=True,
                       timeout=240, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    line = [l for l in p.stdout.splitlines() if l.startswith("AGG")][0].split()
    assert float(line[1]) == 150.0 and abs(float(line[2]) - 2 * 32 * 10 / 0.15) < 1e-6


DDP_WORKER = r'''
import sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/oracle")
from yolov3_b200.parallel import allreduce_gradients, broadcast_parameters, scale_loss, world_size
import torch.nn.functional as F
dist.init_process_group("gloo")
r, W = dist.get_rank(), dist.get_world_size()
torch.manual_seed(100 + r)                      # ranks start different: the broadcast must make them equal
w = torch.randn(8, 4, 3, 3, requires_grad=True); b = torch.randn(8, requires_grad=True)
broadcast_parameters([w, b], 0)
g = torch.Generator().manual_seed(7)
x = torch.randn(6, 4, 10, 10, generator=g); t = torch.randn(6, 8, 10, 10, generator=g)
def shard_loss(xs, ts):                          # reference convention: per-shard mean loss times the shard batch size
    return F.mse_loss(F.conv2d(xs, w, b, padding=1), ts) * xs.shape[0]
lo, hi = r * 3, (r + 1) * 3
scale_loss(shard_loss(x[lo:hi], t[lo:hi])).backward()      # loss *= WORLD_SIZE (train.py:405-406)
allreduce_gradients([w, b])                                  # DDP mean all-reduce
got_w, got_b = w.grad.clone(), b.grad.clone()
w.grad = None; b.grad = None
sum(shard_loss(x[i * 3:(i + 1) * 3], t[i * 3:(i + 1) * 3]) for i in range(W)).backward()   # single-process equivalent
assert torch.allclose(got_w, w.grad, rtol=1e-5, atol=1e-6) and torch.allclose(got_b, b.grad, rtol=1e-5, atol=1e-6)
if r == 0: print("DDP_OK", world_size())
dist.barrier(); dist.destroy_process_group()
'''


def test_ddp_gradient_exchange_semantics_gloo(tmp_path):
    """SURVEY App. D last row: `loss * WORLD_SIZE` + mean all-reduce == sum of the per-rank (loss * bs_rank) gradients."""
    script = tmp_path / "ddp.py"
    script.write_text(DDP_WORKER)
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29654", str(script), str(ROOT)], capture_output=True, text=True,
                       timeout=240, env=dict(os.environ, MASTER_ADDR="127.0.0.1"))
    assert p.returncode == 0, p.stderr[-2000:]
    assert "DDP_OK 2" in p.stdout


def test_autolabel_rows_match_the_reference_semantics():
    """non_max_suppression(labels=...) (utils/general.py:689-695): the adapter appends the priors as obj = 1 / one-hot
    rows; running the ORACLE on that augmented tensor must equal the oracle's own labels= path (which was pinned against
    the reference in tests/golden/make_golden.py)."""
    import numpy as np
    import torch

    import yolo_oracle as O
    from yolov3_b200.nms import _append_labels

    pred = O.synth_predictions(2, n_rows=300, nc=80, seed=4)
    labels = [[[3.0, 320.0, 320.0, 120.0, 90.0]], []]
    aug = _append_labels(pred, labels)
    assert aug.shape == (2, 301, 85) and float(aug[1, 300, 4]) == 0.0 and float(aug[0, 300, 5 + 3]) == 1.0
    a, sa = O.non_max_suppression(aug, 0.25, 0.45)
    b, sb = O.non_max_suppression(pred, 0.25, 0.45, labels=labels)
    for x, y, sx, sy in zip(a, b, sa, sb):
        assert np.array_equal(x, y) and np.array_equal(sx, sy)


def test_xpair_weight_pack_layout():
    """Y3_W_XPAIR (include/yolov3_b200.h): [c_out_pad, 3, 2, 2, c_in] with a zero phantom column."""
    import torch

    from yolov3_b200 import ops

    w = torch.randn(64, 32, 3, 3)
    wp, bp = ops.pack_conv_weight_xpair(w, torch.zeros(64), device="cpu")
    v = wp.float().view(64, 3, 2, 2, 32)
    ref = w.bfloat16().float()
    assert torch.equal(v[:, :, 0, 0], ref[:, :, :, 0].permute(0, 2, 1)) and torch.equal(v[:, :, 0, 1], ref[:, :, :, 1].permute(0, 2, 1))
    assert torch.equal(v[:, :, 1, 0], ref[:, :, :, 2].permute(0, 2, 1)) and float(v[:, :, 1, 1].abs().max()) == 0.0


def test_package_synth_workloads_equal_the_oracle_copies():
    """bench.py / tools draw their synthetic inputs from yolov3_b200.synth (nothing outside tests/, smoke() and the CPU
    baseline leg imports oracle/); the tests use the oracle's generators — both must produce identical tensors."""
    import torch

    import yolo_oracle as O
    from yolov3_b200 import synth

    assert torch.equal(O.synth_predictions(2, n_rows=300, seed=3), synth.synth_predictions(2, n_rows=300, seed=3))
    assert torch.equal(O.synth_targets(16, seed=2), synth.synth_targets(16, seed=2))
    assert O.scaled_hyp() == synth.scaled_hyp() and O.scaled_hyp(nl=2, nc=20, imgsz=320) == synth.scaled_hyp(nl=2, nc=20, imgsz=320)


def test_only_tests_smoke_and_bench_cpu_legs_touch_the_oracle():
    """The oracle is test infrastructure: no file of the package or of tools/ may import it."""
    from pathlib import Path

    root = Path(__file__).resolve().parents[1]
    offenders = []
    for p in list((root / "yolov3_b200").rglob("*.py")) + list((root / "tools").glob("*.py")):
        txt = p.read_text()
        if "yolo_oracle" in txt or "ref_shim" in txt:
            offenders.append(str(p.relative_to(root)))
    assert not offenders, offenders


def _plan(c_in, c_out, k, s, hw, n=32, res=False, head=False, layout=0):
    """y3_conv_plan for a conv of the yolov3 graph: host-only query, fake (aligned, never dereferenced) pointers."""
    import ctypes as C

    from yolov3_b200 import _lib

    L = _lib.lib()
    d = _lib.ConvDesc()
    d.n, d.h, d.w, d.c_in, d.c_out, d.ksize, d.stride, d.act = n, hw, hw, c_in, c_out, k, s, 1
    d.in_, d.in_ld, d.in_coff = 0x10000, c_in, 0
    d.weight, d.bias = 0x20000, 0x30000
    if head:
        d.out_f32, d.out_f32_ld = 0x40000, L.y3_conv_cout_pad(c_out)
    else:
        d.out, d.out_ld, d.out_coff = 0x40000, c_out, 0
    if res:
        d.res, d.res_ld, d.res_coff = 0x50000, c_out, 0
    d.weight_layout = layout
    info = _lib.ConvPlanInfo()
    _lib.check(L.y3_conv_plan(C.byref(d), C.byref(info)), "y3_conv_plan")
    return {k_: getattr(info, k_) for k_, _ in info._fields_}


def test_conv_kernel_selection_for_the_yolov3_layers():
    """The variant conv_tc_prepare picks for the distinct conv shapes of yolov3 @640 bs 32 (SURVEY App. A): tile N = c_out
    bucket, CTA pairs for N >= 128, halo reuse for stride-1 3x3 (N = 256 only as a pair), TMA-store epilogue for stride 1
    except halo + N = 256, resident weights when one N tile's weights fit in 96 KB, two epilogue groups for N <= 128."""
    from yolov3_b200 import _lib

    shapes = [(32, 64, 3, 2, 640, False), (64, 32, 1, 1, 320, False), (32, 64, 3, 1, 320, True), (64, 128, 3, 2, 320, False),
              (128, 64, 1, 1, 160, False), (64, 128, 3, 1, 160, True), (128, 256, 3, 2, 160, False), (256, 128, 1, 1, 80, False),
              (128, 256, 3, 1, 80, True), (256, 512, 3, 2, 80, False), (512, 256, 1, 1, 40, False), (256, 512, 3, 1, 40, True),
              (512, 1024, 3, 2, 40, False), (1024, 512, 1, 1, 20, False), (512, 1024, 3, 1, 20, True), (768, 256, 1, 1, 40, False),
              (384, 128, 1, 1, 80, False)]
    for c_in, c_out, k, s, hw, res in shapes:
        p = _plan(c_in, c_out, k, s, hw, res=res)
        bn = 32 if c_out <= 32 else 64 if c_out <= 64 else 128 if c_out <= 128 else 256
        assert p["block_n"] == bn and p["block_k"] == (64 if c_in % 64 == 0 else 32), (c_in, c_out, p)
        assert p["pair"] == int(bn >= 128) and p["epilogue_groups"] == (2 if bn <= 128 else 1), (c_in, c_out, p)
        assert p["halo"] == int(k == 3 and s == 1), (c_in, c_out, p)
        assert p["staged"] == int(s == 1 and not (p["halo"] and bn == 256)), (c_in, c_out, p)
        n_tiles = -(-c_out // bn)
        w_bytes = k * k * c_in * (bn // 2 if p["pair"] else bn) * 2
        assert p["n_tiles"] == n_tiles and p["resident_weights"] == int(n_tiles == 1 and w_bytes <= 96 * 1024), (c_in, c_out, p)
        if s == 1:
            assert p["m_tiles"] == -(-(32 * (hw + 2) * (hw + 2)) // 128)
        assert 1 <= p["grid"] <= 148 and (p["grid"] % 2 == 0 or not p["pair"])
    # the first stride-2 layer with x-paired weights: 6 taps of 64 channels, one k-block
    d = _plan(32, 64, 3, 2, 640, layout=_lib.W_XPAIR)
    assert d["xpair"] == 1 and d["block_k"] == 64 and d["k_blocks"] == 1 and d["resident_weights"] == 1
    # Detect head: fp32 pixel-major output, never staged
    h = _plan(256, 255, 1, 1, 80, head=True)
    assert h["block_n"] == 256 and h["staged"] == 0 and h["pair"] == 1


def test_reference_arm_json_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): one JSON line with the contract's keys; its
    e2e repeats the value with zero H2D/D2H bytes, cpu_baseline describes the run.  One bounded step on this box's cores."""
    import json
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parents[1]
    # launched the way the driver launches the N > 1 arms (torchrun, one process per GPU): rank 0 alone runs and prints the
    # line, the other rank exits 0 without work and without output
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29671", str(root / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=900, cwd=root,
                       env=dict(os.environ, MASTER_ADDR="127.0.0.1"))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("images/sec @640 bs32 YOLOv3") and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["value"] > 0 and d["n_gpus"] == 2
    assert d["config"]["global_batch"] == 64
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    # the reference's own Model from the staged copy (oracle/_ref) when it is there, else the oracle port — and it says which
    sys.path.insert(0, str(root / "oracle"))
    import ref_shim

    assert d["cpu_baseline"]["kind"] == ("reference" if ref_shim.reference_available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["config"]["batch_per_gpu"] == 32 and "nms" in d


def test_detect_multi_backend_seam():
    """The reference's backend-plugin point (models/common.py:435): same attributes as its ``pt`` branch, loud failure on a
    CPU device, checkpoint dict {"cfg", "state_dict"} accepted."""
    import torch

    from yolov3_b200.backend import DetectMultiBackend, _load
    from yolov3_b200.model import Model

    with pytest.raises(RuntimeError, match="no CPU path"):
        DetectMultiBackend(Model(CFG / "yolov3-tiny.yaml", device="cpu"), device=torch.device("cpu"))
    src = Model(CFG / "yolov3-tiny.yaml", device="cpu")
    m = _load({"cfg": str(CFG / "yolov3-tiny.yaml"), "state_dict": src.state_dict(), "names": ["a"] * 80}, "cpu")
    assert m.names == ["a"] * 80 and all(torch.equal(v, m.state_dict()[k]) for k, v in src.state_dict().items())
    for attr in ("forward", "warmup", "from_numpy", "__call__"):
        assert callable(getattr(DetectMultiBackend, attr))
    # checkpoint round trip through a file
    import tempfile

    from yolov3_b200.backend import save_checkpoint

    with tempfile.TemporaryDirectory() as td:
        save_checkpoint(src, td + "/tiny.pt")
        back = _load(td + "/tiny.pt", "cpu")
    assert back.yaml == src.yaml and all(torch.equal(v, back.state_dict()[k]) for k, v in src.state_dict().items())


def test_package_exports_resolve_to_the_reference_seam_names():
    """`import yolov3_b200` is lazy (no GPU, no library load); every advertised name resolves to the object in its module."""
    import importlib

    import yolov3_b200 as y

    assert set(y.__all__) >= {"Model", "DetectionModel", "DetectMultiBackend", "non_max_suppression", "scale_boxes", "box_iou",
                              "ComputeLoss", "process_batch", "letterbox", "Ensemble", "DDP", "SGD", "ModelEMA", "Pipeline"}
    for name in y.__all__:
        obj = getattr(y, name)
        assert obj is getattr(importlib.import_module(obj.__module__), name)
    with pytest.raises(AttributeError):
        y.no_such_name

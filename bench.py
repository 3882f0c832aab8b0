#!/usr/bin/env python
"""bench.py — BASELINE.json metric on the BASELINE configs, one JSON line on stdout (rank 0).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--only infer,train,spp_nms,nms,lib,cpu]
                  [--dump-outputs DIR]
  torchrun ... bench.py --gpus N ...        (one rank per GPU)

Headline (config 2, `metric`/`value`/`e2e`/`roofline`): a step = one pass of the hot path (Model.forward + Detect decode,
reference models/yolo.py) over one synthetic batch "YOLOv3 640x640 bs=32 inference on 1 B200, synthetic input, random-init
weights"; weak scaling: bs 32 per GPU, no data-path collective.
  value      images/s, inputs resident in HBM (fp32 NCHW), CUDA-graph replay, CUDA-event timing, max over ranks
  e2e        images/s through yolov3_b200.Pipeline with HOST uint8 images: H2D + forward + decode + NMS + D2H per step
  roofline   conv kernels (tensor bound): algorithmic conv FLOPs / event-timed conv_tc launch time, vs MEASURED_PEAKS
  parity_rel_l2   z of the timed bs-32 engine vs the CPU reference/oracle forward on the same images and weights (the run
                  fails above 2e-2)
Extra keys (the other BASELINE configs, tools/bench_workloads.py):
  train      config 4: training step (fwd / loss / bwd + overlapped bucketed all-reduce / fused clip+SGD+EMA), bs 8 per GPU —
             the one path with a collective: its per-N values are the scaling curve of the gradient exchange
  spp_nms    config 3: yolov3-spp forward + decode + NMS(0.25/0.45/1000), bs 8 per GPU, host images in, boxes out
  nms        config 5: five thresholds x single/multi-label on synthetic [32,25200,85]
  gpu_library_baseline   the reference itself on this GPU through PyTorch+cuDNN / torchvision / torch DDP (informational)
  cpu_baseline / --impl reference: the reference's own torch-CPU Model + non_max_suppression from the staged copy
             (oracle/_ref, kind "reference"), else the oracle port (kind "port"), on the host cores, bounded sample.
The timed loop of every leg runs --steps steps.  --dump-outputs DIR writes what the headline's timed forward returned in its last step
(dump_outputs); the inputs and weights are seeded, so two builds run with the same arguments can be compared array by array.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

CFG = "yolov3.yaml"
IMG, BS = 640, 32
GFLOP_PER_IMG = 155.891          # SURVEY §8(d): 2*MAC over the 75 nn.Conv2d of yolov3.yaml @640
GFLOP_LAYER0 = 0.708             # layer 0 runs on CUDA cores (c_in=3); excluded from the tensor roofline
METRIC = "images/sec @640 bs32 YOLOv3"
UNIT = "images/s"
PARITY_TOL = 2e-2
DUMP_ROWS = 65536  # rows of z and of the head logits that --dump-outputs writes: 2 x 22 MB


def peaks():
    from bench_workloads import peaks as _p

    return _p()


def recorded_conv_traffic():
    """`roofline.traffic`: DRAM bytes of the conv_tc launches of ONE forward (bs 32) from the committed ncu capture of
    tools/run_forward.py (profiles/r02_ncu_conv_tc_dram.csv: dram__bytes_read.sum + dram__bytes_write.sum per launch) — a recorded
    capture of the same kernels, not a counter of this run (no profiler runs inside the timed process); null when absent."""
    import csv

    p = ROOT / "profiles" / "r02_ncu_conv_tc_dram.csv"
    if not p.exists():
        return {"traffic": None, "traffic_note": "no committed ncu DRAM capture (profiles/r02_ncu_conv_tc_dram.csv)"}
    try:
        rows = [r for r in csv.DictReader(l for l in p.read_text().splitlines() if not l.startswith("=="))]
        tot, n = 0.0, 0
        for r in rows:
            if r.get("Metric Name") in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                v = float(r["Metric Value"].replace(",", ""))
                v *= {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(r["Metric Unit"], 1)
                tot += v
                n += 1
        launches = n // 2
        return {"traffic": tot, "traffic_unit": "bytes per step (sum over the conv_tc launches of one forward)",
                "traffic_launches": launches, "traffic_source": "profiles/r02_ncu_conv_tc_dram.csv (ncu capture, recorded)"}
    except Exception as e:  # noqa: BLE001
        return {"traffic": None, "traffic_note": f"could not parse the committed capture: {e!r}"}


def workload_config(world):
    return {"workload": f"yolov3.yaml forward+decode, {IMG}x{IMG}, bs {BS}/GPU, random-init weights, folded BN",
            "imgsz": IMG, "batch_per_gpu": BS, "global_batch": BS * world, "parallelism": f"replicas x{world} (no collective)",
            "l2": "inputs larger than L2: two 157 MB fp32 batches alternated; activations 6 GB/step", "cuda_graph": True}


class ClockSampler:
    FIELDS = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    # nvidia-smi needs ~0.2 s to deliver its first line and the timed region of the default run is shorter than that,
    # so the sampler is started before the warm-up, every line is stamped with its arrival time, and stop(t0, t1) keeps
    # the lines that arrived while the GPU ran this workload: the timed region [t0, t1] plus, when that holds fewer than
    # three, the identical untimed replays the caller appends right after it (same graph, same inputs, same clocks)

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append((time.time(), l)) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, l in self.lines:
            if t0 is not None and not (t0 + 0.05 <= ts <= t1 + 0.05):  # a line reports the ~100 ms before it arrived
                continue
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def sample_outputs(z, raw):
    """A fixed, seeded sample of what the timed forward returns: rows of z [bs, rows, 85] (decoded boxes) and the same rows
    of the Detect head's logits p_i [bs, na, ny, nx, 85] (row r of image b in z is decoded from logits row r of image b,
    rows ordered level, anchor, y, x).  ``sample_rows`` holds the flat indices b * rows + r, as float64."""
    import torch

    n, rows, no = z.shape
    idx = torch.randperm(n * rows, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    logits = torch.cat([p.reshape(n, -1, no) for p in raw], 1).reshape(n * rows, no)
    di = idx.to(z.device)
    return {"z": z.reshape(n * rows, no)[di].cpu().numpy(), "raw": logits[di].cpu().numpy(), "sample_rows": idx.double().numpy()}


def dump_outputs(out_dir: Path, arrays):
    import numpy as np

    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a)


def aggregate(ms_local: float, dev) -> float:
    """Max over ranks of a locally event-timed duration (one process per GPU; NCCL on GPUs, gloo in the CPU tests)."""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return ms_local
    t = torch.tensor([ms_local], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def build_model(device):
    import torch

    from yolov3_b200.model import Model

    torch.manual_seed(0)
    m = Model(CFG, device=device)
    # non-trivial BN statistics so that the fold is exercised (SURVEY §8(d) config 2)
    g = torch.Generator().manual_seed(0)
    for k in list(m.params):
        if k.endswith("bn.weight"):
            m.params[k] = torch.rand(m.params[k].shape, generator=g) + 0.5
        elif k.endswith("bn.bias") or k.endswith("running_mean"):
            m.params[k] = torch.randn(m.params[k].shape, generator=g) * 0.1
        elif k.endswith("running_var"):
            m.params[k] = torch.rand(m.params[k].shape, generator=g) + 0.5
    return m


# ------------------------------------------------------------------------------------------ CPU legs (checker / baseline only)
class CpuReference:
    """The reference's torch-CPU forward for the bench model: the reference's OWN ``Model`` from the staged copy
    (oracle/_ref, ``kind = "reference"``) when present, else the oracle port (``kind = "port"``), holding the same weights
    as the GPU model (``params``), fused, fp32, inference mode.  Thread count: calibrated AT the batch that is timed."""

    def __init__(self, params=None):
        import torch

        sys.path.insert(0, str(ROOT / "oracle"))
        import ref_shim
        import yolo_oracle as O

        self.O = O
        self.kind = "port"
        self.nms = None
        if ref_shim.reference_available():
            try:
                ref_shim.install()
                from models.yolo import Model as RefModel
                from utils.general import non_max_suppression as ref_nms

                m = RefModel(str(ref_shim.REFERENCE_ROOT / "models" / CFG))
                if params is not None:
                    missing, unexpected = m.load_state_dict(params, strict=False)
                    assert not unexpected and all("num_batches_tracked" in k for k in missing), (missing[:3], unexpected[:3])
                self.model = m.eval().fuse()
                self.nms = ref_nms
                self.kind = "reference"
            except Exception as e:  # noqa: BLE001  (a broken staged copy must not take the bench down: say so and use the port)
                print(f"bench: staged reference unusable ({e!r}); using the oracle port", file=sys.stderr)
        if self.kind == "port":
            self.model = O.OracleModel(ROOT / "yolov3_b200" / "cfg" / CFG, params=params, seed=0, fused=True)
        self.threads = None
        self.torch = torch

    def forward(self, x):
        with self.torch.inference_mode():
            y = self.model(x)
        return y[0]

    def calibrate(self, x):
        """fastest of {cores, cores/2, cores/4} intra-op threads on THIS batch (one pass each after one warm-up pass)"""
        torch = self.torch
        cores = os.cpu_count() or 1
        best = (None, 1e30)
        tried = {}
        for t in sorted({cores, max(1, cores // 2), max(1, cores // 4)}, reverse=True):
            torch.set_num_threads(t)
            self.forward(x[:2])
            t0 = time.perf_counter()
            self.forward(x)
            dt = time.perf_counter() - t0
            tried[t] = round(x.shape[0] / dt, 2)
            if dt < best[1]:
                best = (t, dt)
        self.threads, self.tried = best[0], tried
        torch.set_num_threads(self.threads)
        return self.threads

    def nms_rate(self, n_img=8, conf=0.25, iou=0.45):
        """reference non_max_suppression on the host cores (config 5).  Called per image: the reference's wall-clock break
        (utils/general.py:675,746-748) would otherwise silently drop the rest of a slow batch."""
        from yolov3_b200.synth import synth_predictions

        pred = synth_predictions(n_img, n_rows=25200, nc=80, seed=3)
        fn = self.nms if self.nms is not None else (lambda p, c, i: self.O.non_max_suppression(p, c, i, use_torchvision=True))
        fn(pred[:1], conf, iou)
        t0 = time.perf_counter()
        for i in range(n_img):
            fn(pred[i:i + 1], conf, iou)
        dt = time.perf_counter() - t0
        return {"input_boxes_per_s": n_img * 25200 / dt, "ms_per_image": dt * 1e3 / n_img, "images": n_img,
                "impl": "reference utils.general.non_max_suppression (torch CPU + torchvision.ops.nms)" if self.nms is not None
                else "oracle candidate pipeline (numpy) + torchvision.ops.nms"}


def run_reference(args, rank):
    """--impl reference: the reference's torch-CPU forward on rank 0's host cores, a bounded sample of each step's batch."""
    if rank != 0:
        return
    import torch

    model = build_model("cpu")  # parameters only: nothing of yolov3_b200's compute path runs in this arm
    ref = CpuReference(params=model.state_dict())
    gen = torch.Generator().manual_seed(1)
    probe = torch.rand(8, 3, IMG, IMG, generator=gen)
    ref.calibrate(probe)
    t0 = time.perf_counter()
    ref.forward(probe)
    rate = 8 / (time.perf_counter() - t0)
    budget = 170.0
    per_step = max(1, min(BS, int(budget / max(1, args.steps + args.warmup) * rate)))
    x = torch.rand(per_step, 3, IMG, IMG, generator=gen)
    for _ in range(args.warmup):
        ref.forward(x)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref.forward(x)
    dt = time.perf_counter() - t0
    v = per_step * args.steps / dt
    try:
        nms_ref = {"conf0.25_iou0.45_single": ref.nms_rate(8, 0.25, 0.45), "conf0.001_iou0.6_single": ref.nms_rate(4, 0.001, 0.6)}
    except Exception as e:  # noqa: BLE001
        nms_ref = {"unavailable": repr(e)[:200]}
    sample = (f"{per_step} of the {BS} images of each step (reference {'Model' if ref.kind == 'reference' else 'forward, oracle port'}, "
              f"fp32, fused BN, torch CPU, {ref.threads} threads of {os.cpu_count()} host cores — img/s by thread count at bs 8: {ref.tried})")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(max(1, args.gpus)),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": ref.threads, "kind": ref.kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "nms": nms_ref,
        "gpu_launches": 0,
    }), flush=True)


# ------------------------------------------------------------------------------------------------ reference on the GPU
def _reference_modules():
    sys.path.insert(0, str(ROOT / "oracle"))
    import ref_shim

    if not ref_shim.reference_available():
        return None
    ref_shim.install()
    return ref_shim


def library_baseline(dev, rank, world, bs=32, img=640, steps=10, train_bs=8):
    """The reference's own code on this GPU through PyTorch's libraries: Model(yolov3.yaml).fuse() in bf16 channels_last
    (cuDNN), utils.general.non_max_suppression (torch ops + torchvision CUDA nms), ComputeLoss + DistributedDataParallel +
    torch.optim.SGD under bf16 autocast.  Informational: this is the bar a kernel library sets on the same hardware."""
    shim = _reference_modules()
    if shim is None:
        return {"unavailable": "reference not staged (oracle/_ref missing: see oracle/stage_reference.py)"}
    from models.yolo import Model as RefModel
    from utils.general import non_max_suppression as ref_nms
    from utils.loss import ComputeLoss as RefLoss

    import torch
    import torch.distributed as dist

    from yolov3_b200 import synth

    res = {"impl": "ultralytics/yolov3 @ 97b87b1 (staged copy) on torch " + torch.__version__ + " / cuDNN " + str(torch.backends.cudnn.version())}
    torch.backends.cudnn.benchmark = True
    cfg = str(shim.REFERENCE_ROOT / "models" / "yolov3.yaml")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        torch.manual_seed(0)
        m = RefModel(cfg).to(dev).eval().fuse().to(torch.bfloat16).to(memory_format=torch.channels_last)
        x = torch.rand(bs, 3, img, img, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        with torch.inference_mode():
            for _ in range(5):
                m(x)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                m(x)
            e1.record()
            torch.cuda.synchronize()
        ms = aggregate(e0.elapsed_time(e1) / steps, dev)
        res["forward"] = {"images_per_s": world * bs / (ms / 1e3), "ms_per_step": ms, "batch_per_gpu": bs,
                          "what": "reference Model.fuse() forward+decode, bf16, channels_last, cuDNN (benchmark mode), resident input"}
        del m, x
    except Exception as e:  # noqa: BLE001
        res["forward"] = {"error": repr(e)[:300]}
    try:
        pred = synth.synth_predictions(bs, n_rows=25200, nc=80, seed=3).to(dev)
        nms = {}
        for conf, iou, ml in ((0.25, 0.45, False), (0.001, 0.6, False), (0.001, 0.6, True)):
            ref_nms(pred[:2], conf, iou, multi_label=ml, max_det=300)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n_done = 0
            for i in range(0, bs, 4):  # 4 images per call keeps the reference's wall-clock break (general.py:746) out of reach
                ref_nms(pred[i:i + 4], conf, iou, multi_label=ml, max_det=300)
                n_done += 4
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            nms[f"conf{conf}_iou{iou}_{'multi' if ml else 'single'}"] = {"input_boxes_per_s": world * n_done * 25200 / dt,
                                                                         "ms_per_batch_of_32": dt * 1e3 * 32 / n_done}
        res["nms"] = {"what": "reference non_max_suppression on the CUDA tensor (torchvision.ops.nms CUDA kernel), wall clock incl. "
                              "its host syncs", **nms}
        del pred
    except Exception as e:  # noqa: BLE001
        res["nms"] = {"error": repr(e)[:300]}
    try:
        torch.manual_seed(0)
        m = RefModel(cfg).to(dev)
        hyp = synth.scaled_hyp()
        m.hyp, m.nc = hyp, 80
        m.train()
        net = m
        if world > 1:
            net = torch.nn.parallel.DistributedDataParallel(m, device_ids=[dev.index], output_device=dev.index)
        opt = torch.optim.SGD(m.parameters(), lr=0.01, momentum=0.937, nesterov=True)
        loss_fn = RefLoss(m)
        x = torch.rand(train_bs, 3, img, img, device=dev)
        targets = synth.synth_targets(train_bs, seed=2 + rank).to(dev)

        def step():
            with torch.autocast("cuda", dtype=torch.bfloat16):
                pred = net(x)
                loss, _ = loss_fn(pred, targets)
                loss = loss * world
            loss.backward()
            torch.nn.utils.clip_grad_norm_(m.parameters(), max_norm=10.0)
            opt.step()
            opt.zero_grad()

        for _ in range(3):
            step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = aggregate(e0.elapsed_time(e1) / steps, dev)
        res["train"] = {"images_per_s": world * train_bs / (ms / 1e3), "ms_per_step": ms, "batch_per_gpu": train_bs,
                        "what": "reference Model + ComputeLoss, torch.autocast(bf16), DistributedDataParallel (NCCL), clip + torch SGD; "
                                "no EMA, no H2D"}
    except Exception as e:  # noqa: BLE001
        res["train"] = {"error": repr(e)[:300]}
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only", default="all", help="comma list of legs besides the headline: train,spp_nms,nms,lib,cpu (default all)")
    ap.add_argument("--per-op", default=None, help="write the per-launch timing table (JSON) to this path")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write a seeded sample of the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    legs = {"train", "spp_nms", "nms", "lib", "cpu"} if args.only == "all" else set(filter(None, args.only.split(","))) - {"none"}
    if args.no_cpu_baseline:
        legs.discard("cpu")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import bench_workloads as W
    from yolov3_b200 import _lib
    from yolov3_b200.pipeline import Pipeline

    model = build_model(dev)
    params_host = model.state_dict()  # for the CPU parity / baseline leg (taken before anything can go wrong on the device)
    eng = model.engine(BS, IMG, IMG, torch.float32)
    n_launch = _lib.lib().y3_model_num_launches(eng.handle)
    # two distinct resident input batches (157 MB each > 126 MB L2), alternated so no step re-reads a cached input.  The first
    # images of batch 0 come from a CPU generator: the parity leg runs the CPU reference on exactly those images.
    n_par = 2
    x_par = torch.rand(n_par, 3, IMG, IMG, generator=torch.Generator().manual_seed(1))
    xs = [torch.rand(BS, 3, IMG, IMG, device=dev, generator=torch.Generator(device=dev).manual_seed(1 + i)) for i in range(2)]
    xs[0][:n_par] = x_par.to(dev)
    graphs = [eng.capture(x) for x in xs]  # one graph per resident input: a step is exactly the 76 launches of a forward

    def step(i):
        graphs[i & 1].replay()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    eng.check_errors()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t_load0 = time.time()
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    dumped = sample_outputs(eng.z, eng.raw) if args.dump_outputs and rank == 0 else None
    clocks = None
    if rank == 0:
        # the clock samples must come from this workload: keep replaying it (untimed) until >= 0.6 s of load were observed
        i = args.steps
        while time.time() - t_load0 < 0.6:
            step(i)
            i += 1
            if i % 8 == 0:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        clocks = sampler.stop(t_load0, time.time())
        clocks["window_s"] = round(time.time() - t_load0, 3)
        clocks["timed_region_s"] = round(ms_total / 1e3, 3)
    ms_total = aggregate(ms_total, dev)
    if world > 1:
        dist.barrier()
    value = world * BS * args.steps / (ms_total / 1e3)
    # output of the timed engine on the parity images (graph 0 = batch 0), kept for the parity leg below
    graphs[0].replay()
    torch.cuda.synchronize()
    eng.check_errors()
    z_par = eng.z[:n_par].detach().cpu().clone()
    z_finite = bool(torch.isfinite(eng.z).all())

    # ---- e2e: host uint8 images -> H2D -> forward -> decode -> NMS -> D2H, through the public Pipeline
    pipe = Pipeline(model, BS, IMG, IMG, conf_thres=0.25, iou_thres=0.45, max_det=300)
    hosts = [torch.randint(0, 256, (BS, 3, IMG, IMG), dtype=torch.uint8, generator=torch.Generator().manual_seed(7 + i)).pin_memory()
             for i in range(2)]
    for i in range(3):
        pipe(hosts[i & 1])
    for _ in pipe.stream(hosts[i & 1] for i in range(3)):
        pass
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    n_det = 0
    for dets in pipe.stream(hosts[i & 1] for i in range(args.steps)):  # every step: H2D of its images, D2H of its boxes
        n_det += sum(d.shape[0] for d in dets)
    e1.record()
    torch.cuda.synchronize()
    ms_e2e = e0.elapsed_time(e1)
    # the synchronous per-batch call (one batch in flight, as the reference's detect.py loop), for comparison
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        pipe(hosts[i & 1])
    torch.cuda.synchronize()
    ms_e2e_sync = (time.perf_counter() - t0) * 1e3
    ms_e2e = aggregate(ms_e2e, dev)
    e2e = world * BS * args.steps / (ms_e2e / 1e3)

    # ---- roofline of the dominant kernel (conv_tc): per-launch CUDA events on the launching stream (rank 0's GPU)
    per_op = None
    if rank == 0:
        from yolov3_b200.profile import time_ops

        per_op = time_ops(eng, xs[0], iters=args.steps)
    del pipe, graphs
    model._engines.clear()
    del eng
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs (every rank takes part: the training step has the collective)
    extra = {}

    def leg(key, fn):
        """An extra leg must never take the headline line down with it: a failure is reported under the leg's key."""
        try:
            extra[key] = fn()
        except Exception as e:  # noqa: BLE001
            print(f"bench: leg '{key}' failed on rank {rank}: {e!r}", file=sys.stderr)
            extra[key] = {"error": repr(e)[:300]}
        try:
            torch.cuda.empty_cache()
        except Exception:  # noqa: BLE001  (a sticky CUDA error: the host-side results above are still valid)
            pass

    if "nms" in legs:
        leg("nms", lambda: {"workload": f"synthetic [bs {BS}/GPU, 25200, 85] fp32 (SURVEY §8d config 5), max_det 300, device-resident, "
                                        "sync-free y3_nms_batched; iou 0.6 at conf <= 0.01 else 0.45", "unit": "input boxes/s",
                            **W.nms_sweep_workload(dev, rank, world, bs=BS, reps=args.steps)})
    if "spp_nms" in legs:
        leg("spp_nms", lambda: W.spp_nms_workload(dev, rank, world, bs=8, img=IMG, steps=args.steps, warmup=args.warmup))
    if "train" in legs:
        leg("train", lambda: W.train_step_workload(dev, rank, world, bs=8, img=IMG, steps=args.steps, warmup=3))
    if "lib" in legs:
        leg("gpu_library_baseline", lambda: library_baseline(dev, rank, world, bs=BS, img=IMG, steps=args.steps))

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    conv_ms = sum(o["ms"] for o in per_op if o["kind"] == "conv_tc")
    all_ms = sum(o["ms"] for o in per_op)
    conv_tflop = (GFLOP_PER_IMG - GFLOP_LAYER0) * BS / 1e3
    pk = peaks()
    achieved = conv_tflop / (conv_ms / 1e3)
    roofline = {"bound": "tensor", "achieved": achieved, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                "frac": achieved / pk["tf_sustained"], "traffic": None,
                "kernel": f"conv_tc_kernel ({sum(1 for o in per_op if o['kind'] == 'conv_tc')} launches/step)",
                "kernel_ms_per_step": conv_ms, "kernel_share_of_step": conv_ms / all_ms,
                "whole_step_frac": GFLOP_PER_IMG * 1e9 * (value / world) / (pk["tf_sustained"] * 1e12),
                "peak_source": pk["source"] + " sustained bf16 (MEASURED_PEAKS.json)",
                **recorded_conv_traffic()}
    dec = [o for o in per_op if o["kind"] == "decode"]
    if dec:  # Detect decode: read the head logits + write z = 17.1 MB/image algorithmic
        roofline["decode_hbm"] = {"bound": "hbm", "achieved": dec[0]["gbs"], "peak": pk["hbm"], "unit": "GB/s",
                                  "frac": dec[0]["gbs"] / pk["hbm"], "ms": dec[0]["ms"]}
    if args.per_op:
        Path(args.per_op).parent.mkdir(parents=True, exist_ok=True)
        Path(args.per_op).write_text(json.dumps(per_op, indent=1))

    cpu, parity = None, None
    if "cpu" in legs:
        ref = CpuReference(params=params_host)
        probe = torch.cat([x_par, torch.rand(6, 3, IMG, IMG, generator=torch.Generator().manual_seed(2))])
        ref.calibrate(probe)
        ref.forward(probe[:2])
        t0 = time.perf_counter()
        z_ref = ref.forward(probe)
        dt = time.perf_counter() - t0
        cpu = {"value": probe.shape[0] / dt, "unit": UNIT, "cores": ref.threads, "kind": ref.kind,
               "sample": f"8 of the {BS} images of a step, one timed pass after warm-up and thread calibration "
                         f"(img/s by thread count: {ref.tried}); "
                         + ("reference models.yolo.Model from oracle/_ref" if ref.kind == "reference" else "oracle port")}
        zr = z_ref[:n_par].double()
        parity = float((z_par.double() - zr).norm() / zr.norm())

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": workload_config(world),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity_rel_l2": parity, "parity": {"what": f"z[:{n_par}] of the timed bs-{BS} CUDA-graph engine vs the CPU {cpu['kind'] if cpu else 'reference'} "
                                                    "forward on the same images and weights", "tolerance": PARITY_TOL, "z_all_finite": z_finite},
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": BS * 3 * IMG * IMG, "d2h_bytes_per_step": BS * 300 * 6 * 4 + 2 * BS * 4,
                "ms_per_step": ms_e2e / args.steps, "path": "Pipeline.stream: uint8 H2D -> forward -> decode -> NMS(0.25/0.45/300) -> D2H, two batches in flight",
                "sync_call_ms_per_step": ms_e2e_sync / args.steps},
        "gpu_launches": n_launch * args.steps,
        "clocks": clocks,
        **extra,
    }
    if dumped is not None:
        dump_outputs(Path(args.dump_outputs), dumped)
    print(json.dumps(line), flush=True)
    if not z_finite or (parity is not None and not parity <= PARITY_TOL):
        print(f"bench: PARITY FAILURE: rel-L2 {parity} (tolerance {PARITY_TOL}), finite {z_finite}", file=sys.stderr)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        sys.exit(3)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

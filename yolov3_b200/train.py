"""Training-mode forward + backward of the YOLOv3 graph on the sm_100a kernels (SURVEY §8 rows a19/a20).

Mirrors what the reference runs in ``train.py:401-411`` — ``pred = model(imgs)`` in train mode (BatchNorm with batch
statistics, eps 1e-3 / momentum 0.03; ``Detect`` returning the raw ``[bs,na,ny,nx,no]`` maps, models/yolo.py:110), then
``loss.backward()`` through every Conv block — without autograd graphs or cuDNN:

  forward  per Conv block:  conv (tcgen05 implicit GEMM, identity epilogue) -> bn_stats (per-block partial sums)
                            -> bn_finalize (fixed-order second stage, running statistics) -> bn_act_fwd
  backward per Conv block:  bn_act_bwd (partial sums -> dgamma/dbeta accumulated into the flat gradient buffer -> dy)
                            -> wgrad (tcgen05, accumulating straight into the parameter's .grad view)
                            -> dgrad, which is the SAME conv kernel run on dy with the transposed, tap-flipped weight pack
                               (stride-2 layers: on the zero-stuffed dy), accumulating into the input's gradient through
                               the residual port (the Bottleneck shortcut's gradient rides on that port too).

Parameters, gradients and the bf16 weight copy live in ONE flat buffer each (``params.ParamStore``): the forward re-packs
all weights with two launches, the backward writes every gradient in place, and the data-parallel exchange all-reduces
contiguous ranges of the gradient buffer on a side stream while the remaining layers are still being back-propagated
(``parallel.DDP``; reference: DistributedDataParallel buckets, utils/torch_utils.py:60-72).  Every reduction is two-stage
with a fixed summation order — no floating-point atomics — except the split-K wgrad (``deterministic=True`` removes that too)
and the loss (csrc/y3_loss.cu): it adds the dL/dp of matches that share a cell with float atomics, so on a cell with three
or more matches the last bits of that gradient depend on the order the adds land in, and it sums its loss terms with
double atomics before rounding them to float.

``TrainEngine.forward/backward`` are wrapped in one ``torch.autograd.Function`` so that the reference's
``loss.backward(); optimizer.step()`` work unchanged on the fp32 master parameters (``Model.parameters()``).
Supported layer types in train mode: Conv, Bottleneck, SPP, nn.Upsample, Concat, Detect (= yolov3.yaml, yolov3-spp.yaml).
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.distributed as dist

from . import _lib, ops
from . import train_ops as T
from .tensors import PaddedNHWC, _stream


def _wide(t: PaddedNHWC) -> PaddedNHWC:
    """The >= 32-channel view of a 16-channel slice (its buffer was allocated 32 wide with a zero upper half)."""
    return t if t.c >= 32 else PaddedNHWC(t.buf, t.coff, 32)


class _Block:
    """One Conv+BN+SiLU block (models/common.py:57-81) with everything its forward and backward need."""

    __slots__ = ("prefix", "c1", "c2", "k", "s", "x", "y", "a", "res", "upsample", "wf", "wd", "st", "dw", "first", "dy",
                 "dy_up", "post_fwd", "pre_bwd", "gamma", "beta", "rmean", "rvar", "dgamma", "dbeta", "nblk")


class TrainEngine:
    use_graphs = True        # replay forward / backward segments as CUDA graphs after one eager warm-up step
    deterministic = False    # True: wgrad without split-K (bit-reproducible steps; slower on the early layers)
    n_buckets = 4            # gradient ranges all-reduced separately, each as soon as its layers are done
    dgrad_phases = True      # stride-2 dgrad as four parity-class convs of the un-stuffed dy (False: conv of the zero-stuffed dy)

    def __init__(self, model, n, h, w, keep_all=False):
        """keep_all=True gives every block its own dy buffer (per-layer gradient checks in the tests); the default shares
        one scratch buffer per shape."""
        dev = model.device
        self.model, self.n, self.h, self.w = model, n, h, w
        det = model.detect
        nodes = model.nodes
        gs = int(max(det.stride.tolist()))
        if h % gs or w % gs:  # same rule as the inference Engine (utils/general.py:281-292 check_img_size)
            raise ValueError(f"image size {h}x{w} must be a multiple of the max stride {gs}")
        self.fwd_gen = 0  # activations live in this engine's buffers: a backward must belong to the LAST forward
        for nd in nodes[:-1]:
            if nd.type not in ("Conv", "Bottleneck", "Upsample", "Concat", "SPP", "MaxPool2d", "ZeroPad2d"):
                raise NotImplementedError(f"training-mode {nd.type} is not built")
        store = model.store()
        self.store = store
        self.P = model.device_params()
        self.world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        self.sync_bn = bool(getattr(model, "sync_bn", False)) and self.world > 1
        if self.sync_bn:
            self.use_graphs = False  # the per-layer collectives stay eager launches
        self.blocks: list[_Block] = []
        self.keep = []
        self.grad_bufs: dict[int, PaddedNHWC] = {}
        self.scratch: dict[tuple, PaddedNHWC] = {}
        self.keep_all = keep_all
        self.zero_bias = torch.zeros(4096, dtype=torch.float32, device=dev)  # identity-epilogue convs (forward and dgrad)
        max_partial = 0

        def buf(c, hh, ww, ld=None):
            # the conv kernel produces multiples of 32 output channels: a 16-channel tensor (yolov3-tiny layers 0-2) lives in a
            # 32-channel buffer whose upper half stays zero (zero weight rows / zero dgrad rows), everything else sees c = 16
            b = PaddedNHWC.zeros(n, hh, ww, c, device=dev, ld=max(ld or c, 32))
            self.keep.append(b)
            return b

        def f32(c):
            t = torch.zeros(c, dtype=torch.float32, device=dev)
            self.keep.append(t)
            return t

        def new_block(prefix, c1, c2, k, s, x, a, res=None, upsample=False, first=False):
            nonlocal max_partial
            b = _Block()
            b.prefix, b.c1, b.c2, b.k, b.s, b.x, b.a, b.res, b.upsample, b.first = prefix, c1, c2, k, s, x, a, res, upsample, first
            ho, wo = x.h // s, x.w // s
            b.y = buf(c2, ho, wo)
            b.wf = store.weight_rows_bf16(prefix + ".conv.weight")
            b.wd = None if first else torch.zeros(ops.cout_pad(c1), k * k * c2, dtype=torch.bfloat16, device=dev)
            b.dw = store.grad_rows(prefix + ".conv.weight")
            b.gamma, b.beta = store.flat(prefix + ".bn.weight"), store.flat(prefix + ".bn.bias")
            b.dgamma, b.dbeta = store.flat(prefix + ".bn.weight", grad=True), store.flat(prefix + ".bn.bias", grad=True)
            b.rmean, b.rvar = store.flat(prefix + ".bn.running_mean"), store.flat(prefix + ".bn.running_var")
            b.st = {name: f32(c2) for name in ("scale", "shift", "mean", "rstd")}
            b.st.update(sums=f32(2 * c2), gsums=f32(2 * c2))  # [sum | sumsq] forward, [sum dz | sum dz*xhat] backward
            b.nblk = T.partial_blocks(n, ho, wo, c2)
            max_partial = max(max_partial, b.nblk * 2 * c2)
            b.dy = buf(c2, ho, wo) if keep_all else self._scratch(c2, ho, wo, dev)
            b.dy_up = self._scratch(c2, x.h, x.w, dev, tag="up") if s == 2 else None
            b.post_fwd, b.pre_bwd = [], []  # extra launches after this block's forward / before its backward (SPP pools)
            self.blocks.append(b)
            return b

        # ---- shapes and concat destinations (same zero-copy concat / fused upsample layout as the inference engine)
        shp = {}
        for nd in nodes[:-1]:
            src = [(model.ch, h, w) if s < 0 else shp[s] for s in nd.srcs]
            c0, h0, w0 = src[0]
            if nd.type == "Conv":
                s_ = nd.args[3] if len(nd.args) > 3 else 1
                shp[nd.i] = (nd.c_out, h0 // s_, w0 // s_)
            elif nd.type in ("Bottleneck", "SPP"):
                shp[nd.i] = (nd.c_out, h0, w0)
            elif nd.type == "Upsample":
                shp[nd.i] = (c0, h0 * 2, w0 * 2)
            elif nd.type == "Concat":
                shp[nd.i] = (sum(s[0] for s in src), h0, w0)
            elif nd.type == "ZeroPad2d":
                shp[nd.i] = (c0, h0, w0)  # virtual: folded into the MaxPool2d(2,1,0) that follows (out-of-bounds = 0)
            elif nd.type == "MaxPool2d":
                k_, s2_ = nd.args[0], (nd.args[1] if len(nd.args) > 1 else nd.args[0])
                shp[nd.i] = (c0, h0, w0) if (k_, s2_) == (2, 1) else (c0, h0 // s2_, w0 // s2_)
        consumers = {}
        for nd in nodes:
            for s in nd.srcs:
                consumers.setdefault(s, []).append(nd.i)
        cat_buf, alias, up_alias = {}, {}, {}
        for nd in nodes[:-1]:
            if nd.type != "Concat":
                continue
            c, hh, ww = shp[nd.i]
            cat = buf(c, hh, ww)
            cat_buf[nd.i] = cat
            off = 0
            for s in nd.srcs:
                cs = shp[s][0]
                sl = cat.slice(off, cs)
                off += cs
                if nodes[s].type == "Upsample":
                    v = nodes[s].srcs[0]
                    assert consumers.get(v) == [s] and consumers.get(s) == [nd.i] and nodes[v].type == "Conv"
                    up_alias[v] = sl
                else:
                    alias[s] = sl

        def out_of(i):
            if i in alias:
                return alias[i]
            c, hh, ww = shp[i]
            return buf(c, hh, ww)

        # ---- lower the graph into Conv blocks
        self.im2col = buf(32, h, w)
        tens = {}
        for nd in nodes[:-1]:
            srcs = [tens[s] if s >= 0 else None for s in nd.srcs]
            base = f"model.{nd.i}"
            reps = [base] if nd.n == 1 else [f"{base}.{j}" for j in range(nd.n)]
            if nd.type == "Conv":
                c1, c2, *rest = nd.args
                k = rest[0] if len(rest) > 0 else 1
                s_ = rest[1] if len(rest) > 1 else 1
                x = srcs[0]
                for ri, r in enumerate(reps):
                    last = ri == len(reps) - 1
                    if x is None:
                        assert c1 == 3 and k == 3 and s_ == 1
                        a = out_of(nd.i) if last else buf(c2, h, w)
                        new_block(r, 32, c2, 1, 1, self.im2col, a, first=True)  # layer 0 = 1x1 conv over the im2col
                    elif last and nd.i in up_alias:
                        a = up_alias[nd.i]
                        new_block(r, c1, c2, k, s_, x, a, upsample=True)
                    else:
                        a = out_of(nd.i) if last else buf(c2, x.h // s_, x.w // s_)
                        new_block(r, c1, c2, k, s_, x, a)
                    x = a
                tens[nd.i] = x
            elif nd.type == "Bottleneck":
                c1, c2, *rest = nd.args
                shortcut = rest[0] if rest else True
                x = srcs[0]
                c_ = int(c2 * 0.5)
                for ri, r in enumerate(reps):
                    yb = out_of(nd.i) if ri == len(reps) - 1 else buf(c2, x.h, x.w)
                    t = buf(c_, x.h, x.w)
                    new_block(r + ".cv1", c1, c_, 1, 1, x, t)
                    new_block(r + ".cv2", c_, c2, 3, 1, t, yb, res=x if (shortcut and c1 == c2) else None)
                    x, c1 = yb, c2
                tens[nd.i] = x
            elif nd.type == "SPP":
                # models/common.py:281-290: cv2(cat[x, mp5(x), mp9(x), mp13(x)]) with x = cv1(input); each pool reads x
                c1, c2, *rest = nd.args
                ks = tuple(rest[0]) if rest else (5, 9, 13)
                x = srcs[0]
                c_ = c1 // 2
                cat = buf((len(ks) + 1) * c_, x.h, x.w)
                b1 = new_block(base + ".cv1", c1, c_, 1, 1, x, cat.slice(0, c_))
                for q, k in enumerate(ks):
                    idx = torch.zeros(n * x.h * x.w * c_, dtype=torch.uint8, device=dev)
                    self.keep.append(idx)
                    src, dst = cat.slice(0, c_), cat.slice((q + 1) * c_, c_)
                    b1.post_fwd.append(lambda src=src, dst=dst, k=k, idx=idx: T.maxpool_train_fwd(src, dst, k, idx))
                    b1.pre_bwd.append(lambda src=src, dst=dst, k=k, idx=idx: T.maxpool_bwd(self.grad_of(dst), self.grad_of(src),
                                                                                        k, idx, accumulate=True))
                y = out_of(nd.i)
                new_block(base + ".cv2", (len(ks) + 1) * c_, c2, 1, 1, cat, y)
                tens[nd.i] = y
            elif nd.type == "Upsample":
                tens[nd.i] = None
            elif nd.type == "Concat":
                tens[nd.i] = cat_buf[nd.i]
            elif nd.type == "ZeroPad2d":  # yolov3-tiny.yaml:29: nn.ZeroPad2d([0,1,0,1]) feeding nn.MaxPool2d(2,1,0)
                assert tuple(nd.args[0]) == (0, 1, 0, 1) and all(nodes[c].type == "MaxPool2d" for c in consumers.get(nd.i, []))
                tens[nd.i] = ("zeropad", srcs[0])
            elif nd.type == "MaxPool2d":
                k = nd.args[0]
                s_ = nd.args[1] if len(nd.args) > 1 else k
                pd = nd.args[2] if len(nd.args) > 2 else 0
                x, oob_zero = srcs[0], False
                if isinstance(x, tuple):
                    assert (k, s_, pd) == (2, 1, 0), "only ZeroPad2d([0,1,0,1]) + MaxPool2d(2,1,0)"
                    x, oob_zero = x[1], True
                y = out_of(nd.i)
                idx = torch.zeros(n * y.h * y.w * x.c, dtype=torch.uint8, device=dev)
                self.keep.append(idx)
                host = self.blocks[-1]  # the pool runs after the latest block's forward and before that block's backward
                host.post_fwd.append(lambda x=x, y=y, k=k, s_=s_, pd=pd, idx=idx, oz=oob_zero:
                                     T.maxpool_train_fwd(x, y, k, idx, stride=s_, off=-pd, oob_zero=oz))
                host.pre_bwd.append(lambda x=x, y=y, k=k, s_=s_, pd=pd, idx=idx: self._pool_backward(x, y, k, s_, -pd, idx))
                tens[nd.i] = y

        # ---- Detect heads
        self.heads = []
        head_ld = ops.cout_pad(det.na * det.no)
        dec = _lib.DecodeDesc()
        for j, s in enumerate(nodes[-1].srcs):
            x = tens[s]
            wname, bname = f"model.{det.i}.m.{j}.weight", f"model.{det.i}.m.{j}.bias"
            hd = dict(x=x, c1=x.c, j=j, wname=wname, bname=bname)
            hd["out"] = torch.zeros(n * x.h * x.w, head_ld, dtype=torch.float32, device=dev)
            hd["raw"] = torch.zeros(n, det.na, x.h, x.w, det.no, dtype=torch.float32, device=dev)
            hd["wf"] = store.weight_rows_bf16(wname)                   # [256, c1]: row 255 is the zero pad row of the slot
            hd["wd"] = torch.zeros(ops.cout_pad(x.c), head_ld, dtype=torch.bfloat16, device=dev)
            hd["bias"] = store.flat(bname, padded=True)[:head_ld]      # fp32 master bias read in place (pad entry = 0)
            hd["dy"] = buf(head_ld, x.h, x.w)
            hd["dw"] = store.grad_rows(wname)                          # [256, 1, c1]
            hd["db"] = store.flat(bname, grad=True, padded=True)[:head_ld]
            hd["nblk"] = T.partial_blocks(n, x.h)
            max_partial = max(max_partial, hd["nblk"] * 256)
            self.heads.append(hd)
            lv = dec.levels[j]
            lv.head, lv.head_ld, lv.raw_out = hd["out"].data_ptr(), head_ld, hd["raw"].data_ptr()
            lv.ny, lv.nx, lv.stride = x.h, x.w, float(det.stride[j])
        dec.nl, dec.bs, dec.na, dec.no, dec.z = det.nl, n, det.na, det.no, None
        self.dec = dec
        self.err = torch.zeros(1, dtype=torch.int32, device=dev)
        self.partial = torch.zeros(max_partial, dtype=torch.float32, device=dev)  # first-stage rows of every reduction

        # ---- one table for the batched dgrad re-pack (y3_pack_dgrad_batched)
        items, tile = [], 0
        for hd in self.heads:
            s = store.slots[hd["wname"]]
            items.append((s.offset, hd["wd"], s.rows, s.ci, 1, head_ld))
        for b in self.blocks:
            if b.wd is not None:
                s = store.slots[b.prefix + ".conv.weight"]
                items.append((s.offset, b.wd, s.rows, s.ci, b.k, b.c2))
        arr = (_lib.PackItem * len(items))()
        for i, (off, dst, rows, ci, k, dst_co) in enumerate(items):
            it = arr[i]
            rows = min(rows, dst_co)
            it.src_off, it.dst, it.co_rows, it.ci, it.k, it.dst_co, it.tile_begin = off, dst.data_ptr(), rows, ci, k, dst_co, tile
            tile += k * k * ((rows + 31) // 32) * ((ci + 31) // 32)
        self.pack_items = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(dev)
        self.n_pack_items, self.pack_tiles = len(items), tile

        self.param_names = []
        for b in self.blocks:
            self.param_names += [b.prefix + ".conv.weight", b.prefix + ".bn.weight", b.prefix + ".bn.bias"]
        for hd in self.heads:
            self.param_names += [hd["wname"], hd["bname"]]

        # ---- backward segments: [heads + last blocks | ... | first blocks], cut where the gradient buckets end
        self.buckets = store.bucket_ranges(self.n_buckets)
        ends = [e for _, e in self.buckets]
        self.segments: list[list[_Block]] = [[] for _ in ends]
        si = 0
        for b in reversed(self.blocks):
            off = store.slots[b.prefix + ".conv.weight"].offset
            while off >= ends[si]:
                si += 1
            self.segments[si].append(b)
        self.comm = None          # side stream of the gradient exchange (parallel.DDP)
        self._graphs: dict = {}

    # ------------------------------------------------------------------------------------------------ helpers
    def _scratch(self, c, hh, ww, dev, tag=""):
        key = (c, hh, ww, tag)
        if key not in self.scratch:
            self.scratch[key] = PaddedNHWC.zeros(self.n, hh, ww, c, device=dev)
        return self.scratch[key]

    def grad_of(self, t: PaddedNHWC) -> PaddedNHWC:
        """Gradient buffer mirroring an activation buffer (same geometry, same channel slice)."""
        key = t.buf.data_ptr()
        g = self.grad_bufs.get(key)
        if g is None:
            g = self.grad_bufs[key] = PaddedNHWC(torch.zeros_like(t.buf), 0, t.buf.shape[3])
        return g.slice(t.coff, t.c)

    def _run(self, key, fn):
        """Run ``fn`` eagerly the first time (function attributes, lazy allocations), capture AND replay it the second time,
        replay it afterwards.  Every launch inside is stream-ordered with no host synchronisation and all buffers keep their
        addresses."""
        if not self.use_graphs:
            return fn()
        st = self._graphs.setdefault(key, {"n": 0})
        if st["n"] == 0:
            st["n"] = 1
            return fn()
        if "graph" not in st:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                st["out"] = fn()
            st["graph"] = g
        st["graph"].replay()
        return st["out"]

    # ------------------------------------------------------------------------------------------------ forward
    def forward(self, x: torch.Tensor, in_div=0.0):
        self.fwd_gen += 1
        if not self.use_graphs:
            return self._forward_impl(x, in_div)
        st = self._graphs.setdefault("fwd", {"n": 0})
        if st["n"] == 0:
            st["n"] = 1
            return self._forward_impl(x, in_div)
        if "graph" not in st:
            st["x"], st["div"] = x.clone(), in_div
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                st["out"] = self._forward_impl(st["x"], in_div)
            st["graph"] = g
        assert in_div == st["div"] and x.shape == st["x"].shape and x.dtype == st["x"].dtype
        st["x"].copy_(x)
        st["graph"].replay()
        return st["out"]

    def refresh_packs(self):
        """bf16 forward packs (views of the flat bf16 copy) and dgrad packs from the current fp32 masters: two launches."""
        s = self.store
        T.f32_to_bf16(s.P[:s.n_train], s.Wbf)
        T.pack_dgrad_batched(self.pack_items, self.n_pack_items, s.Wbf, self.pack_tiles)

    def _forward_impl(self, x: torch.Tensor, in_div=0.0):
        det = self.model.detect
        self.refresh_packs()
        T.im2col_first(x, self.im2col, in_div)
        zb = self.zero_bias
        for b in self.blocks:
            ops.conv_bn_act(b.x, b.wf, zb, max(b.c2, 32), b.k, b.s, ops.ACT_NONE, out=_wide(b.y), err=self.err)
            st = b.st
            T.bn_stats(b.y, self.partial)
            count = self.n * b.y.h * b.y.w
            if self.sync_bn:  # nn.SyncBatchNorm (train.py:270-272): batch statistics over every rank's pixels
                T.colreduce(self.partial, b.nblk, 2 * b.c2, st["sums"])
                dist.all_reduce(st["sums"])  # [sum | sumsq] share one buffer: one collective per layer
                T.bn_finalize(st["sums"], 1, b.gamma, b.beta, count * self.world, st["scale"], st["shift"], st["mean"],
                              st["rstd"], b.rmean, b.rvar)
            else:
                T.bn_finalize(self.partial, b.nblk, b.gamma, b.beta, count, st["scale"], st["shift"], st["mean"], st["rstd"],
                              b.rmean, b.rvar)
            T.bn_act_fwd(b.y, st["scale"], st["shift"], b.a, b.res, b.upsample)
            for fn in b.post_fwd:
                fn()
        co = det.na * det.no
        for hd in self.heads:
            ops.conv_bn_act(hd["x"], hd["wf"], hd["bias"], co, 1, 1, ops.ACT_NONE, out_f32=hd["out"], err=self.err)
        _lib.check(_lib.lib().y3_detect_head_decode_fwd(C.byref(self.dec), _stream()), "y3_detect_head_decode_fwd")
        return [hd["raw"] for hd in self.heads]

    # ------------------------------------------------------------------------------------------------ backward
    def backward(self, graws):
        """graws: dL/draw per level (fp32 [n,na,ny,nx,no]).  Gradients are ACCUMULATED into the flat gradient buffer
        (``store.G``; zeroed first unless earlier gradients are live, like autograd's .grad semantics) and attached to the
        parameters as ``.grad`` views.  With ``parallel.DDP`` enabled, each gradient bucket is all-reduced on a side stream as
        soon as the segment producing it has been enqueued."""
        store = self.store
        if not store.grads_are_live():
            store.G.zero_()
        ddp = getattr(self.model, "ddp", None)
        exchange = ddp is not None and ddp.require_sync and self.world > 1
        if exchange and self.comm is None:
            # high priority: the all-reduce CTAs take the SMs the persistent conv / wgrad grids release first
            self.comm = torch.cuda.Stream(device=self.model.device, priority=-1)
        main = torch.cuda.current_stream()
        if self.use_graphs:
            st = self._graphs.setdefault("bwd_in", {})
            if "g" not in st:
                st["g"] = [g.detach().float().contiguous().clone() for g in graws]
            for dst, src in zip(st["g"], graws):
                dst.copy_(src)
            graws = st["g"]
        else:
            graws = [g.detach().float().contiguous() for g in graws]
        self._written, self._pending_res, self._pending_add = set(), {}, {}
        for si, seg in enumerate(self.segments):
            self._run(("bwd", si), lambda si=si, seg=seg: self._backward_segment(si, seg, graws))
            if exchange:
                lo, hi = self.buckets[si]
                ev = torch.cuda.Event()
                ev.record(main)
                self.comm.wait_event(ev)
                with torch.cuda.stream(self.comm):
                    dist.all_reduce(store.G[lo:hi], op=dist.ReduceOp.SUM)
        if exchange:
            main.wait_stream(self.comm)
            ddp.pending_average = True  # G holds SUMS over ranks: the optimizer folds 1/world into its update, or
            #                             parallel.DDP.finish() divides in place for a plain torch.optim optimizer
        store.attach_grads()

    def _contribute_conv(self, dy, wd, c_in, k, x, s2=False):
        gx = _wide(self.grad_of(x))  # c_in = 16: the dgrad conv writes 32 channels, the upper 16 from zero weight rows
        c_in = max(c_in, 32)
        key = (x.buf.data_ptr(), x.coff, x.c)
        first = key not in self._written and not self._overlaps(self._written, key)
        pend = self._pending_res.pop(key, None)

        def conv(res):
            if s2:
                ops.conv_dgrad_s2(dy, wd, self.zero_bias, c_in, out=gx, res=res, err=self.err)
            else:
                ops.conv_bn_act(dy, wd, self.zero_bias, c_in, k, 1, ops.ACT_NONE, out=gx, res=res, err=self.err)

        if first:
            # the Bottleneck shortcut's gradient (da of the block that added x) rides on the residual port of this dgrad
            conv(pend)
        else:
            conv(gx)
            if pend is not None:
                T.add_nhwc(pend, gx, accumulate=True)
        self._written.add(key)

    def _pool_backward(self, x, y, k, stride, off, idx):
        """grad(x) (+)= gather of grad(y) through the recorded argmax; first contribution writes, later ones accumulate."""
        key = (x.buf.data_ptr(), x.coff, x.c)
        first = key not in self._written and not self._overlaps(self._written, key)
        T.maxpool_bwd(self.grad_of(y), self.grad_of(x), k, idx, accumulate=not first, stride=stride, off=off)
        self._written.add(key)

    def _flush_pending(self):
        for key, (src, dst) in list(self._pending_add.items()):
            first = key not in self._written and not self._overlaps(self._written, key)
            T.add_nhwc(src, self.grad_of(dst), accumulate=not first)
            self._written.add(key)
            self._pending_res.pop(key, None)
        self._pending_add.clear()

    def _backward_segment(self, si, seg, graws):
        det = self.model.detect
        det_flag = 1 if self.deterministic else 0
        if si == 0:
            for hd, g in zip(self.heads, graws):
                x = hd["x"]
                T.head_grad_pack(g, hd["dy"], self.partial)
                T.colreduce(self.partial, hd["nblk"], 256, hd["db"], accumulate=True)
                T.conv_wgrad(hd["dy"], x, hd["dw"], 1, layout=_lib.DW_OHWI, accumulate=True, deterministic=det_flag)
                self._contribute_conv(hd["dy"], hd["wd"], hd["c1"], 1, x)
        for b in seg:
            st = b.st
            for fn in b.pre_bwd:
                fn()
            da = self.grad_of(b.a)
            if self.sync_bn:
                # local sums are the (rank-local) gamma/beta gradients; dy needs the sums over all ranks
                T.bn_act_bwd(b.y, da, b.dy, st, st["sums"], self.partial, b.dbeta, b.dgamma, b.upsample, phase=1)
                st["gsums"].copy_(st["sums"])
                dist.all_reduce(st["gsums"])
                T.bn_act_bwd(b.y, da, b.dy, st, st["gsums"], None, None, None, b.upsample, phase=2,
                             count=self.n * b.y.h * b.y.w * self.world)
            else:
                T.bn_act_bwd(b.y, da, b.dy, st, st["sums"], self.partial, b.dbeta, b.dgamma, b.upsample)
            src = b.dy
            direct_w = b.s == 2 and T.wgrad_s2_supported(b.x.h, b.x.w)
            if b.s == 2 and not (direct_w and self.dgrad_phases):
                src = T.zero_stuff(b.dy, b.dy_up)  # fallback: stride-1 formulations on the zero-stuffed dy
            if direct_w:
                # wgrad straight from the un-stuffed dy (x through its parity view): a quarter of the pixels, no zeros multiplied
                T.conv_wgrad(b.dy, b.x, b.dw, b.k, layout=_lib.DW_OHWI, accumulate=True, deterministic=det_flag, stride=2)
            else:
                T.conv_wgrad(src, b.x, b.dw, b.k, layout=_lib.DW_OHWI, accumulate=True, deterministic=det_flag)
            if b.res is not None:
                # Bottleneck shortcut: the block output's gradient also flows to its input.  It is folded into the next
                # dgrad into that tensor (cv1 of the same Bottleneck: the very next block) through the residual port, or
                # added by a separate launch if no such dgrad arrives before the segment ends.
                self._flush_pending()
                r = b.res
                key = (r.buf.data_ptr(), r.coff, r.c)
                self._pending_res[key] = da
                self._pending_add[key] = (da, r)
            if not b.first:
                key = (b.x.buf.data_ptr(), b.x.coff, b.x.c)
                if b.s == 2 and self.dgrad_phases:
                    # transposed stride-2 conv by parity classes on the un-stuffed dy (4 launches, a quarter of the MMA work)
                    self._contribute_conv(b.dy, b.wd, b.c1, b.k, b.x, s2=True)
                else:
                    self._contribute_conv(src, b.wd, b.c1, b.k, b.x)
                self._pending_add.pop(key, None)
        self._flush_pending()  # a segment is one CUDA graph: nothing may stay pending across its end
        return None

    @staticmethod
    def _overlaps(written, key):
        ptr, coff, c = key
        return any(p == ptr and not (coff + c <= o or o + cc <= coff) for (p, o, cc) in written)

    def check_errors(self):
        e = int(self.err.item())
        if e:
            raise _lib.Y3Error(f"device watchdog reported pipeline stall code {e}")


class TrainFn(torch.autograd.Function):
    """pred = model(imgs) in train mode as ONE autograd node: backward() runs TrainEngine.backward, which leaves every
    parameter gradient in the flat gradient buffer and attaches the ``.grad`` views itself (autograd sees None)."""

    @staticmethod
    def forward(ctx, engine, x, in_div, *params):
        ctx.engine = engine
        raws = engine.forward(x, in_div)
        ctx.gen = engine.fwd_gen
        ctx.n_params = len(params)
        return tuple(r.clone() for r in raws)

    @staticmethod
    def backward(ctx, *graws):
        if ctx.gen != ctx.engine.fwd_gen:
            raise RuntimeError("backward() of a train-mode forward whose activations were overwritten by a later forward of the "
                               "same shape: call loss.backward() before the next model(imgs) (one forward in flight per shape)")
        ctx.engine.backward(graws)
        return (None, None, None) + (None,) * ctx.n_params

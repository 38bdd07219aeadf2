"""Two-stream model builder: the ``Model`` / ``Detect`` / ``parse_model`` surface of the reference's
models/yolo_test.py, built on the icafusion_b200 operator classes.

``Model(cfg, ch=3, nc=None)`` accepts the reference's YAML row format (``[from, number, module, args]``) or a
stock name; ``model(rgb, ir)`` returns what the reference returns (eval: ``(z, logits, [x0,x1,x2])``).
The walk over the layer list follows Model.forward_once (yolo_test.py:136-163) -- ``f == -4`` routes the IR
image -- but runs on NHWC tensors and issues the RGB and IR streams as *grouped* launches (one kernel, two
filter banks), since both streams have identical geometry.
"""
from __future__ import annotations

import logging
import math
from copy import deepcopy
from typing import List

import torch
import torch.nn as nn

from . import ops
from .cfg import load_cfg
from .common import (C3, SPPF, Bottleneck, Concat, Conv, TransformerFusionBlock, Upsample, to_nchw, to_nhwc)
from .ops import ACT_NONE

logger = logging.getLogger(__name__)

_MODULES = {"Conv": Conv, "C3": C3, "SPPF": SPPF, "Bottleneck": Bottleneck, "Concat": Concat,
            "nn.Upsample": Upsample, "Upsample": Upsample, "TransformerFusionBlock": TransformerFusionBlock}


def make_divisible(x, divisor):
    """reference: utils/general.py:234-236"""
    return math.ceil(x / divisor) * divisor


class Detect(nn.Module):
    """Detection head (reference: models/yolo_test.py:26-70): per level a 1x1 Conv2d to na*(nc+5) channels,
    reshaped to (B,na,ny,nx,no); in eval additionally sigmoid + grid/anchor decode, concatenated over levels."""
    stride = None
    export = False

    def __init__(self, nc=80, anchors=(), ch=()):
        super().__init__()
        self.nc = nc
        self.no = nc + 5
        self.nl = len(anchors)
        self.na = len(anchors[0]) // 2
        self.grid = [torch.zeros(1)] * self.nl
        a = torch.tensor(anchors).float().view(self.nl, -1, 2)
        self.register_buffer("anchors", a)
        self.register_buffer("anchor_grid", a.clone().view(self.nl, 1, -1, 1, 1, 2))
        self.m = nn.ModuleList(nn.Conv2d(x, self.no * self.na, 1) for x in ch)

    def _packed(self, i):
        conv = self.m[i]
        key = (conv.weight.data_ptr(), conv.weight._version, conv.bias.data_ptr(), conv.bias._version)
        cache = self.__dict__.setdefault("_icaf_pack", {})
        if i not in cache or cache[i][0] != key:
            cache[i] = (key, ops.pack_conv_weight(conv.weight, conv.bias, 1, 0, ACT_NONE))
        return cache[i][1]

    def alloc_outputs(self, B: int, level_hw, device):
        """(z, logits, row offsets) for levels of spatial sizes level_hw = [(ny, nx), ...]."""
        rows = [self.na * ny * nx for ny, nx in level_hw]
        total = sum(rows)
        z = torch.empty(B, total, self.no, dtype=torch.float16, device=device)
        logits = torch.empty(B, total, self.no - 5, dtype=torch.float16, device=device)
        offs = [sum(rows[:i]) for i in range(len(rows))]
        return z, logits, offs

    def run_level(self, i: int, v: torch.Tensor, z, logits, off: int):
        """One detection level: 1x1 conv (yolo_test.py:49) + decode (:50-63) into rows [off, off+na*ny*nx) of z/logits."""
        if self.training:
            raise NotImplementedError("Detect.run_level is the inference path (decode); in train() call Detect.forward / autograd.detect")
        ag = self.anchor_grid
        key = (ag.data_ptr(), ag._version, ag.device)
        cache = self.__dict__.get("_icaf_anchor_px")
        if cache is None or cache[0] != key:       # host copy of anchor_grid (pixels); re-read when the buffer changes
            cache = (key, ag.detach().float().cpu().view(self.nl, -1).tolist())
            self.__dict__["_icaf_anchor_px"] = cache
        anchor_px = cache[1]
        p = ops.conv2d([v], [self._packed(i)])[0]
        return ops.detect_decode(p, self.na, self.no, z, logits, off, float(self.stride[i]), anchor_px[i])

    def run(self, vs: List[torch.Tensor]):
        """vs: NHWC maps of the nl levels."""
        z, logits, offs = self.alloc_outputs(vs[0].shape[0], [(v.shape[1], v.shape[2]) for v in vs], vs[0].device)
        xs = [self.run_level(i, v, z, logits, offs[i]) for i, v in enumerate(vs)]
        return z, logits, xs

    def forward(self, x):
        if self.training:                                  # yolo_test.py:49-51: the raw maps only
            from . import autograd
            return autograd.detect(self, [to_nhwc(t) for t in x])
        z, logits, xs = self.run([to_nhwc(t) for t in x])
        for i in range(self.nl):
            x[i] = xs[i]                 # the reference overwrites its input list in place (yolo_test.py:49-51)
        return z, logits, x


def check_anchor_order(m: "Detect") -> None:
    """Anchor areas must grow with the stride; flip the levels if the YAML lists them the other way round
    (reference: utils/autoanchor.py:12-20, called from Model.__init__, yolo_test.py:106)."""
    if m.anchor_grid.device.type == "meta":       # shape-only construction (torch.device("meta")): nothing to compare
        return
    a = m.anchor_grid.prod(-1).view(-1)
    if (a[-1] - a[0]).sign() != (m.stride[-1] - m.stride[0]).sign():
        m.anchors[:] = m.anchors.flip(0)
        m.anchor_grid[:] = m.anchor_grid.flip(0)


def fuse_conv_and_bn(conv: nn.Conv2d, bn: nn.BatchNorm2d) -> nn.Conv2d:
    """Fold an eval-mode BatchNorm into the preceding bias-free convolution
    (same result as the reference's utils/torch_utils.py:182-202)."""
    fused = nn.Conv2d(conv.in_channels, conv.out_channels, conv.kernel_size, conv.stride, conv.padding,
                      groups=conv.groups, bias=True).requires_grad_(False).to(conv.weight.device, conv.weight.dtype)
    with torch.no_grad():
        scale = (bn.weight / torch.sqrt(bn.running_var + bn.eps)).to(conv.weight.dtype)
        fused.weight.copy_(conv.weight * scale.view(-1, 1, 1, 1))
        b = conv.bias if conv.bias is not None else torch.zeros_like(bn.running_mean)
        fused.bias.copy_((b - bn.running_mean) * scale + bn.bias)
    return fused


def parse_model(d: dict, ch: List[int]):
    """Build the layer list from YAML rows (reference: models/yolo_test.py:216-302; the subset of module
    types the Transfusion configurations use)."""
    anchors, nc, gd, gw = d["anchors"], d["nc"], d["depth_multiple"], d["width_multiple"]
    na = (len(anchors[0]) // 2) if isinstance(anchors, list) else anchors
    no = na * (nc + 5)
    layers, save, c2 = [], [], ch[-1]
    for i, (f, n, m, args) in enumerate(d["backbone"] + d["head"]):
        name = m if isinstance(m, str) else m.__name__
        if name == "Detect":
            cls = Detect
        elif name in _MODULES:
            cls = _MODULES[name]
        else:
            raise NotImplementedError(f"parse_model: module '{name}' is outside the ICAFusion hot path built here")
        args = [nc if a == "nc" else anchors if a == "anchors" else (None if a == "None" else a) for a in args]
        n = max(round(n * gd), 1) if n > 1 else n
        if cls in (Conv, C3, SPPF, Bottleneck):
            c1 = 3 if (cls is Conv and args[0] == 64) else ch[f]      # yolo_test.py:242-246: both stems take an image
            c2 = args[0]
            if c2 != no:
                c2 = make_divisible(c2 * gw, 8)
            args = [c1, c2, *args[1:]]
            if cls is C3:
                args.insert(2, n)
                n = 1
        elif cls is Concat:
            c2 = sum(ch[x] for x in f)
        elif cls is Detect:
            args.append([ch[x] for x in f])
            if isinstance(args[1], int):
                args[1] = [list(range(args[1] * 2))] * len(f)
        elif cls is TransformerFusionBlock:
            c2 = ch[f[0]]
            args = [c2, *args[1:]]
        else:   # Upsample
            c2 = ch[f]
        m_ = nn.Sequential(*[cls(*args) for _ in range(n)]) if n > 1 else cls(*args)
        t = f"{cls.__module__}.{cls.__name__}"
        np_ = sum(x.numel() for x in m_.parameters())
        m_.i, m_.f, m_.type, m_.np = i, f, t, np_
        logger.info("%3s%18s%3s%10.0f  %-40s%-30s" % (i, f, n, np_, t, args))
        save.extend(x % i for x in ([f] if isinstance(f, int) else f) if x != -1)
        layers.append(m_)
        if i == 0:
            ch = []
        ch.append(c2)
    return nn.Sequential(*layers), sorted(save)


class Model(nn.Module):
    """reference: models/yolo_test.py:73-213"""

    def __init__(self, cfg="yolov5s_Transfusion_kaist", ch=3, nc=None, anchors=None):
        super().__init__()
        self.yaml = load_cfg(cfg)
        ch = self.yaml["ch"] = self.yaml.get("ch", ch)
        if nc and nc != self.yaml["nc"]:
            logger.info(f"Overriding model.yaml nc={self.yaml['nc']} with nc={nc}")
            self.yaml["nc"] = nc
        if anchors:
            self.yaml["anchors"] = round(anchors)
        self.model, self.save = parse_model(deepcopy(self.yaml), ch=[ch])
        self.names = [str(i) for i in range(self.yaml["nc"])]
        m = self.model[-1]
        if isinstance(m, Detect):
            m.stride = torch.Tensor([8.0, 16.0, 32.0])              # yolo_test.py:104 (hard-coded in the reference)
            m.anchors /= m.stride.view(-1, 1, 1)
            check_anchor_order(m)
            self.stride = m.stride
        for mod in self.modules():                                    # utils/torch_utils.py:144-154
            if type(mod) is nn.BatchNorm2d:
                mod.eps = 1e-3
                mod.momentum = 0.03
        self._plan_streams()
        self._plan_concats()

    # -- two-stream pairing ----------------------------------------------------------------------
    def _plan_streams(self):
        """Find the IR stream (first layer with from == -4) and check it mirrors the RGB stream layer by layer."""
        layers = list(self.model)
        starts = [m.i for m in layers if m.f == -4]
        self._ir_start = None
        if len(starts) != 1:
            return
        s = starts[0]
        if 2 * s > len(layers):
            return
        def sig(m):
            return (type(m), [tuple(p.shape) for p in m.parameters()])
        for k in range(s):
            a, b = layers[k], layers[s + k]
            if sig(a) != sig(b) or (k > 0 and (a.f != -1 or b.f != -1)):
                return
        self._ir_start = s

    def _plan_concats(self):
        """Concat elimination: every tensor that feeds a Concat layer is produced directly inside that layer's output
        buffer (all kernels take channel-slice views), so Concat itself launches nothing.  Maps producer layer index ->
        (concat layer index, channel offset); a producer feeding two concats keeps the first and is copied for the rest."""
        self._concat_dst, self._concat_width = {}, {}
        ch = self._layer_ch = {}
        paired = 2 * self._ir_start if self._ir_start is not None else 0     # stream layers run in the grouped loop
        for m in self.model:
            if isinstance(m, Concat) and m.d == 1 and isinstance(m.f, (list, tuple)):
                srcs = [m.i - 1 if j == -1 else j for j in m.f]
                ok = all(j in ch and ch[j] and j >= paired and j not in self._concat_dst and
                         not isinstance(self.model[j], (Concat, Detect)) for j in srcs)
                if ok:
                    off = 0
                    for j in srcs:
                        self._concat_dst[j] = (m.i, off)
                        off += ch[j]
                    self._concat_width[m.i] = off
            ch[m.i] = self._out_channels(m, ch)

    @staticmethod
    def _out_channels(m, ch):
        if isinstance(m, Conv):
            return m.conv.out_channels
        if isinstance(m, (C3,)):
            return m.cv3.conv.out_channels
        if isinstance(m, SPPF):
            return m.cv2.conv.out_channels
        if isinstance(m, TransformerFusionBlock):
            return m.n_embd
        if isinstance(m, nn.Upsample):
            return ch[m.i - 1] if m.f == -1 else ch[m.f]
        if isinstance(m, Concat):
            return sum(ch[m.i - 1 if j == -1 else j] for j in m.f)
        return None

    def forward(self, x, x2, augment=False, profile=False):
        if augment:
            raise NotImplementedError("augmented (multi-scale / flip) inference is outside the hot path built here")
        if tuple(x.shape) != tuple(x2.shape):
            raise ValueError(f"RGB and IR batches must share one shape, got {tuple(x.shape)} and {tuple(x2.shape)}")
        smax = int(self.stride.max()) if hasattr(self, "stride") else 32
        if x.dim() != 4 or x.shape[2] % smax or x.shape[3] % smax:
            # the reference fails at torch.cat for such inputs (models/common.py:321); here the concat buffers are planned
            # from the stride pyramid, so reject up front
            raise ValueError(f"image height and width must be multiples of the maximum stride {smax}, got {tuple(x.shape)}")
        return self.forward_once(x, x2, profile)

    def forward_once(self, x, x2, profile=False):
        if self.training:                           # train.py:336: the list of raw Detect maps, with an autograd graph
            from . import autograd
            return autograd.model_forward(self, x, x2)
        z, logits, xs = self._forward_nhwc(x, x2)
        return z, logits, xs

    def _run_layer(self, m, v, out=None):
        o = None if out is None else [out]
        if isinstance(m, Conv):
            return Conv.run([m], [v], o)[0]
        if isinstance(m, C3):
            return C3.run([m], [v], o)[0]
        if isinstance(m, SPPF):
            return SPPF.run([m], [v], o)[0]
        if isinstance(m, nn.Upsample):             # ours, or torch's own class inside an unpickled reference checkpoint
            if m.mode != "nearest" or m.scale_factor is None or float(m.scale_factor) != 2.0:
                raise NotImplementedError("Upsample: only nearest x2 is supported")
            return ops.upsample2x(v, out)
        if isinstance(m, Concat):
            return Concat.run(v)
        if isinstance(m, TransformerFusionBlock):
            return m.run(v[0], v[1], out)
        if isinstance(m, Detect):
            return m.run(list(v))
        raise NotImplementedError(type(m).__name__)

    def _stage(self, img, stem):
        """Image staging for the stem layer `stem` (a Conv taking the 3-channel image)."""
        if img.dim() != 4 or img.shape[1] != 3:
            raise ValueError(f"expected (B,3,H,W) images, got {tuple(img.shape)}")
        if not ops.on_device(img):
            raise RuntimeError("icafusion_b200 runs on CUDA tensors only (no CPU fallback)")
        if isinstance(stem, Conv) and stem.conv.in_channels == 3:
            return stem.stage_image(img)
        if img.dtype not in (torch.float16, torch.float32, torch.uint8):
            img = img.float()
        return ops.pack_image(img, 1.0 / 255.0 if img.dtype == torch.uint8 else 1.0)

    def _side_streams(self, device, n: int):
        pool = self.__dict__.setdefault("_icaf_streams", {})
        lst = pool.setdefault(device, [])
        while len(lst) < n:
            lst.append(torch.cuda.Stream(device))
        return lst

    def _forward_nhwc(self, rgb, ir):
        """Layer walk with branch-level concurrency: the RGB/IR streams run as grouped launches on the current stream;
        a DMFF block is forked onto a side stream as soon as both of its inputs exist (P3 and P4 fusion overlap the rest of
        the backbone), Detect levels are forked as soon as their head output exists; consumers join before they read."""
        if "_ir_start" not in self.__dict__:       # an unpickled checkpoint (models/experimental.py:118) never ran __init__
            self._plan_streams()
            self._plan_concats()
        layers = list(self.model)
        y: List = [None] * len(layers)
        dev = rgb.device
        if not ops.on_device(rgb):
            raise RuntimeError("icafusion_b200 runs on CUDA tensors only (no CPU fallback)")
        dry = ops.dry_running()                   # shape-only walk on meta tensors (no streams, nothing launched)
        main = None if dry else torch.cuda.current_stream(dev)
        forked = {}                               # layer index -> side stream its result is being produced on
        n_side = [0]
        concurrent = self.__dict__.get("_icaf_concurrent", True) and not dry

        def fork():
            st = self._side_streams(dev, n_side[0] + 1)[n_side[0]]
            n_side[0] += 1
            st.wait_stream(main)
            return st

        def join(idxs):
            for j in idxs:
                st = forked.pop(j, None)
                if st is not None:
                    main.wait_stream(st)

        cats = {}                                 # concat layer index -> its (lazily allocated) output buffer

        def dest(m, shape_hw):
            """Slice of the consumer Concat's buffer this layer should write into (or None)."""
            d = self._concat_dst.get(m.i)
            if d is None:
                return None
            ci, off = d
            if ci not in cats:
                B, H, W = shape_hw
                cats[ci] = torch.empty(B, H, W, self._concat_width[ci], dtype=torch.float16, device=dev)
            return cats[ci][..., off:off + self._layer_ch[m.i]]

        arena = self.__dict__.get("_icaf_arena")
        if concurrent and arena is not None and arena.numel() * 2 <= (96 << 20):
            # the whole packed filter set fits the 126 MB L2: stream it in once, concurrently with the first layers
            st = fork()
            with torch.cuda.stream(st):
                ops.prefetch_l2(arena)
            forked[("prefetch",)] = st
        ir_first = next((m for m in layers if m.f == -4), layers[0])
        v_rgb, v_ir = self._stage(rgb, layers[0]), self._stage(ir, ir_first)
        start = 0
        if self._ir_start is not None:
            s = self._ir_start
            fusion = [m for m in layers[2 * s:] if isinstance(m, TransformerFusionBlock) and isinstance(m.f, (list, tuple))
                      and all(0 <= j < 2 * s for j in m.f)]
            a, b = v_rgb, v_ir
            for k in range(s):                       # both streams, one grouped launch per operator
                ma, mb = layers[k], layers[s + k]
                run = Conv.run if isinstance(ma, Conv) else C3.run if isinstance(ma, C3) else SPPF.run
                a, b = run([ma, mb], [a, b])
                y[k], y[s + k] = a, b
                if concurrent:
                    for m in fusion[:-1]:            # the last fusion block feeds the head directly: it stays in order
                        if y[m.i] is None and all(y[j] is not None for j in m.f):
                            xa, xb = y[m.f[0]], y[m.f[1]]
                            out = dest(m, (xa.shape[0], xa.shape[1], xa.shape[2]))     # allocated on the main stream
                            st = fork()
                            with torch.cuda.stream(st):
                                y[m.i] = m.run(xa, xb, out)
                            forked[m.i] = st
            start = 2 * s
            x = b
        else:
            x = v_rgb

        det = layers[-1] if isinstance(layers[-1], Detect) and isinstance(layers[-1].f, (list, tuple)) else None
        det_state = None
        for m in layers[start:]:
            if y[m.i] is not None and m.i in forked or (y[m.i] is not None and isinstance(m, TransformerFusionBlock)):
                x = y[m.i]                         # already produced (possibly still in flight on a side stream)
                continue
            srcs = [m.i - 1] if m.f == -1 else ([] if m.f == -4 else ([m.f] if isinstance(m.f, int) else
                                                                         [m.i - 1 if j == -1 else j for j in m.f]))
            if m.f == -4:
                x = v_ir
            elif m.f != -1:
                x = y[m.f] if isinstance(m.f, int) else [x if j == -1 else y[j] for j in m.f]
            if m is det and concurrent and det_state is not None:
                # levels whose inputs were ready were forked earlier; run the rest here and join everything
                z, logits, offs, xs = det_state
                for i, j in enumerate(m.f):
                    if xs[i] is None:
                        join([j])
                        xs[i] = m.run_level(i, y[j], z, logits, offs[i])
                for st in list(forked.values()):
                    main.wait_stream(st)
                forked.clear()
                x = (z, logits, xs)
                y[m.i] = x
                continue
            join(srcs)
            if isinstance(m, Concat) and m.i in cats:
                join([j for j, (ci, _) in self._concat_dst.items() if ci == m.i])
                x = cats[m.i]                      # every source already wrote its slice
            else:
                out = None
                if m.i in self._concat_dst and not isinstance(m, (Concat, Detect)):
                    ref = x[0] if isinstance(x, (list, tuple)) else x
                    B, H, W = ref.shape[0], ref.shape[1], ref.shape[2]
                    if isinstance(m, nn.Upsample):
                        H, W = 2 * H, 2 * W
                    elif isinstance(m, Conv):
                        k, s_, p = m.conv.kernel_size[0], m.conv.stride[0], m.conv.padding[0]
                        H, W = (H + 2 * p - k) // s_ + 1, (W + 2 * p - k) // s_ + 1
                    out = dest(m, (B, H, W))
                x = self._run_layer(m, x, out)
            y[m.i] = x
            # fork Detect levels as soon as their input exists (all but the last one, which closes the forward)
            if det is not None and concurrent and m.i in det.f and m.i != det.f[-1] and not isinstance(x, (list, tuple)):
                if det_state is None:
                    B = x.shape[0]
                    Himg, Wimg = rgb.shape[2], rgb.shape[3]
                    hw = [(int(Himg // float(st_)), int(Wimg // float(st_))) for st_ in det.stride]
                    z, logits, offs = det.alloc_outputs(B, hw, dev)
                    det_state = (z, logits, offs, [None] * det.nl)
                i = det.f.index(m.i)
                z, logits, offs, xs = det_state
                if (x.shape[1], x.shape[2]) == (int(rgb.shape[2] // float(det.stride[i])), int(rgb.shape[3] // float(det.stride[i]))):
                    st = fork()
                    with torch.cuda.stream(st):
                        xs[i] = det.run_level(i, x, z, logits, offs[i])
                    forked[("det", i)] = st
        for st in forked.values():                 # nothing may outlive the forward on a side stream
            main.wait_stream(st)
        return x

    def consolidate_weights(self, rgb, ir):
        """Run one forward on (rgb, ir), collect every packed filter it touches and move them into one contiguous arena
        (enables the per-step L2 prefetch).  Call again after the parameters change (re-packing creates new tensors)."""
        with ops.trace_weights() as tr:
            self._forward_nhwc(rgb, ir)
        self.__dict__["_icaf_arena"] = ops.consolidate_weights(tr.items)
        return self.__dict__["_icaf_arena"]

    def fuse(self):
        """Fold every Conv's BatchNorm (reference: models/yolo_test.py:182-190)."""
        for m in self.model.modules():
            if type(m) is Conv and hasattr(m, "bn"):
                m.conv = fuse_conv_and_bn(m.conv, m.bn)
                delattr(m, "bn")
                m.forward = m.fuseforward
                m.__dict__.pop("_icaf_pack", None)
        return self

    def info(self, verbose=False, img_size=640):
        n_p = sum(x.numel() for x in self.parameters())
        logger.info(f"Model Summary: {len(list(self.modules()))} layers, {n_p} parameters")

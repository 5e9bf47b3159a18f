"""Execution engine: BN-folded packed weights + the kernel schedule of ``CABiNet.forward``.

Host side of the hot path.  It owns no arithmetic: every tensor op of the reference forward
(``src/models/cabinet.py:207-247`` and everything it calls) is one of the C-ABI entry points of
``libcabinet_b200.so``; PyTorch is used for device memory (caching allocator), the current stream
and parameter storage only.

Layout: activations are NHWC in HBM, bf16 (``precision='bf16'``) or fp32 (``'fp32'`` parity mode);
class-logit maps at 1/32 and 1/8 resolution and all GAP/SE statistics stay fp32.  Concatenations
(``torch.cat`` at cabinet.py:87,143) are never materialised by a copy: producers write channel
slices of one wider buffer through their pixel stride.
"""

from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import ACT_HSIGMOID, ACT_HSWISH, ACT_NONE, ACT_RELU, ACT_SIGMOID, BF16, F16, F32, check
from .constants import BN_EPS


_DTYPE_CODES = {torch.float32: F32, torch.bfloat16: BF16, torch.float16: F16}


def dtype_code(dtype: torch.dtype) -> int:
    """C-ABI element-type code of a tensor dtype; any other dtype is an error, never passed on as fp32."""
    code = _DTYPE_CODES.get(dtype)
    if code is None:
        raise TypeError(f"cabinet_b200 kernels take float32, bfloat16 or float16 tensors, got {dtype}")
    return code


@dataclass
class Map:
    """A (N,H,W,C) NHWC view: base tensor kept alive + pointer/stride bookkeeping."""

    t: torch.Tensor
    N: int
    H: int
    W: int
    C: int
    ld: int
    off: int = 0  # channel offset inside the pixel
    needs_grad: bool = False  # training step: the map depends on a parameter that requires grad

    @property
    def dt(self) -> int:
        return dtype_code(self.t.dtype)

    @property
    def ptr(self) -> int:
        return self.t.data_ptr() + self.off * self.t.element_size()

    def slice(self, c0: int, c: int) -> "Map":
        return Map(self.t, self.N, self.H, self.W, c, self.ld, self.off + c0, self.needs_grad)

    def nhwc(self) -> torch.Tensor:
        """Dense torch view (tests/debug)."""
        return self.t.view(self.N, self.H, self.W, self.ld)[..., self.off:self.off + self.C]


def _host(t):
    """Parameter -> fp32 CPU tensor.  Folding / packing is a few hundred tiny tensor ops: done once on the host (one
    D2H per parameter) instead of ~900 elementwise kernel launches, then uploaded (`Engine._pack`)."""
    return t.detach().float().cpu()


def _fold(conv_w, conv_b, bn, eps=BN_EPS):
    """Conv + eval-BN -> (w', b') in fp32: y = conv(x, w') + b'  (fold before any rounding)."""
    w = _host(conv_w)
    cout = w.shape[0]
    if bn is None:
        b = _host(conv_b).clone() if conv_b is not None else torch.zeros(cout)
        return w, b
    scale = _host(bn.weight) / torch.sqrt(_host(bn.running_var) + eps)
    b = _host(bn.bias) - _host(bn.running_mean) * scale
    if conv_b is not None:
        b = b + _host(conv_b) * scale
    return w * scale.view(-1, 1, 1, 1), b


class ConvLayer:
    """Dense conv (+folded BN) packed for the kernels: w [Cout][KH*KW*Cin] (c fastest), fp32 bias."""

    def __init__(self, conv, bn, act, wdtype, name="", folded=None):
        if folded is not None:  # (w [Cout,Cin,KH,KW] fp32, b [Cout] fp32, stride, pad): weights derived at pack time
            w, b, self.stride, self.pad = folded
        else:
            w, b = _fold(conv.weight, conv.bias, bn)
            self.stride, self.pad = conv.stride[0], conv.padding[0]
        self.name = name
        self.cout, self.cin, self.kh, self.kw = w.shape
        self.act = act
        self.w = w.permute(0, 2, 3, 1).reshape(self.cout, -1).contiguous().to(wdtype)
        self.b = b.contiguous()
        self.tc = None  # tcgen05 packing: bf16 [ceil16(Cout)][taps][ceil64(Cin)], zero padded
        if wdtype == torch.bfloat16 and self.stride in (1, 2):
            n16, c64, taps = -(-self.cout // 16) * 16, -(-self.cin // 64) * 64, self.kh * self.kw
            pk = torch.zeros((n16, taps, c64), dtype=torch.float32, device=w.device)
            pk[: self.cout, :, : self.cin] = w.permute(0, 2, 3, 1).reshape(self.cout, taps, self.cin)
            self.tc = pk.to(torch.bfloat16).contiguous()


class DwLayer:
    """Depthwise conv (+folded BN): w [k*k][C] fp32, bias fp32."""

    def __init__(self, conv, bn, act, name=""):
        w, b = _fold(conv.weight, conv.bias, bn)
        self.name = name
        self.c, self.k, self.stride, self.act = w.shape[0], w.shape[2], conv.stride[0], act
        self.w = w.view(self.c, -1).t().contiguous()
        self.b = b.contiguous()


class GateLayer:
    """SE (Linear/Linear + hard-sigmoid) or FFM (1x1/1x1 + sigmoid) channel gate, fp32."""

    def __init__(self, w1, b1, w2, b2, gate):
        f = lambda t: None if t is None else _host(t).reshape(t.shape[0], -1).contiguous()  # noqa: E731
        self.w1, self.w2 = f(w1), f(w2)
        self.b1 = None if b1 is None else _host(b1).contiguous()
        self.b2 = None if b2 is None else _host(b2).contiguous()
        self.cmid, self.c = self.w1.shape
        self.gate = gate


_LAYER_TYPES = {c.__name__: c for c in (ConvLayer, DwLayer, GateLayer)}


def _to_plain(o):
    """Layer objects -> tagged dicts of their attributes (recursively); containers and tensors pass through."""
    if type(o).__name__ in _LAYER_TYPES:
        return {"__layer__": type(o).__name__, "vars": {k: _to_plain(v) for k, v in vars(o).items()}}
    if isinstance(o, dict):
        return {k: _to_plain(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return type(o)(_to_plain(v) for v in o)
    return o


def _map_tensors(o, fn):
    """Apply ``fn`` to every tensor inside layers / dicts / lists / tuples (layer objects are updated in place)."""
    if isinstance(o, torch.Tensor):
        return fn(o)
    if type(o).__name__ in _LAYER_TYPES:
        for k, v in vars(o).items():
            setattr(o, k, _map_tensors(v, fn))
        return o
    if isinstance(o, dict):
        return {k: _map_tensors(v, fn) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return type(o)(_map_tensors(v, fn) for v in o)
    return o


def _from_plain(o):
    if isinstance(o, dict):
        if "__layer__" in o:
            obj = object.__new__(_LAYER_TYPES[o["__layer__"]])
            obj.__dict__.update({k: _from_plain(v) for k, v in o["vars"].items()})
            return obj
        return {k: _from_plain(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return type(o)(_from_plain(v) for v in o)
    return o


def _nchw_strides(t: torch.Tensor):
    """(n, y, x, c) element strides of an NCHW tensor, in the order ``Engine.relayout`` takes them."""
    return (t.stride(0), t.stride(2), t.stride(3), t.stride(1))


def _out_size(n, k, s, p):
    return (n + 2 * p - k) // s + 1


def backbone_hw(specs, H: int, W: int) -> Tuple[int, int]:
    """(h, w) of the backbone's output for a stem output of H x W: the stride-2 depthwise convolutions of the blocks
    (``MBConv.spec`` dicts; padding (k - 1) / 2)."""
    for s in specs:
        if s["s"] == 2:
            H, W = _out_size(H, s["k"], 2, (s["k"] - 1) // 2), _out_size(W, s["k"], 2, (s["k"] - 1) // 2)
    return H, W


def _stem_tc2_pack(pk, bias, b_hi):
    """cabinet_stem_tc2 / cabinet_stem7_tc weights from ``pk`` [n][3][7 ky][8 kx] fp32 (kx = 0 zero): W[o][ky][kx][c] (c = 3:
    the constant-1 channel, carrying the bias -- ``b_hi`` its bf16 part -- at the centre pixel) as UMMA core matrices
    [ky][K half][k chunk][o][8]."""
    n = pk.shape[0]
    wn = torch.zeros((n, 7, 8, 4), dtype=torch.float32, device=pk.device)
    wn[..., :3] = pk.permute(0, 2, 3, 1)
    wn[:, 3, 4, 3], wn[:, 3, 5, 3] = b_hi, bias - b_hi
    return wn.view(n, 7, 2, 2, 8).permute(1, 2, 3, 0, 4).contiguous().to(torch.bfloat16)


class Engine:
    # everything ``_pack`` produces (what ``checkpoint.save_packed`` caches)
    PACKED_ATTRS = ("stem", "blocks", "last", "stem_tc", "sb1", "sb2", "sb3", "sb4", "conva", "to_q", "to_k", "to_v",
                    "psp_k", "psp_v", "proj_out", "local", "gamma", "convb", "b1", "b4", "key_ch", "qkv", "ffm_blk",
                    "ffm_gate", "head_conv", "head_out", "ffm_sb", "low_fold", "stem_tc2")
    # what ``_pack_cab`` produces: all an engine built over a standalone ContextAggregationBlock packs
    CAB_ATTRS = ("to_q", "to_k", "to_v", "psp_k", "psp_v", "proj_out", "local", "gamma", "key_ch", "qkv")
    # what ``_pack_mobilenet`` produces: all an engine built over a standalone MobileNetV3 packs
    BACKBONE_ATTRS = ("stem", "blocks", "last", "stem_tc3")
    # ... and what an engine over a standalone SpatialBranch / AttentionBranch / FeatureFusionModule / CABiNetOutput packs
    SB_ATTRS = ("sb1", "sb2", "sb3", "sb4", "stem_tc7")
    AB_ATTRS = ("conva", "convb", "b1", "b4") + CAB_ATTRS
    FFM_ATTRS = ("ffm_blk", "ffm_gate")
    HEAD_ATTRS = ("head_conv", "head_out")

    def __init__(self, model, precision: str = "bf16", packed: Optional[dict] = None):
        if precision not in ("bf16", "fp32"):
            raise ValueError(f"precision must be 'bf16' or 'fp32', got {precision!r}")
        p0 = next(model.parameters())
        if not p0.is_cuda:
            raise RuntimeError("cabinet_b200 engine needs the model on a CUDA device (no CPU path)")
        from . import modules

        self.lib = _lib.load()
        self.dev = p0.device
        self.precision = precision
        self.tdt = torch.bfloat16 if precision == "bf16" else torch.float32
        self.dt = BF16 if precision == "bf16" else F32
        # an engine over a standalone module packs that module alone (``attrs``) and runs its ``forward_*`` method:
        # ContextAggregationBlock -> forward_block, MobileNetV3 -> forward_backbone, SpatialBranch -> forward_sb,
        # AttentionBranch -> forward_ab, FeatureFusionModule -> forward_ffm, CABiNetOutput -> forward_head
        # (subclasses included: a user's subclass with its own forward packs and runs as its base class)
        standalone = None
        for cls, v in ((modules.ContextAggregationBlock, (self._pack_cab, self.CAB_ATTRS)),
                       (modules.MobileNetV3, (self._pack_mobilenet, self.BACKBONE_ATTRS)),
                       (modules.SpatialBranch, (self._pack_spatial, self.SB_ATTRS)),
                       (modules.AttentionBranch, (self._pack_ab, self.AB_ATTRS)),
                       (modules.FeatureFusionModule, (self._pack_ffm, self.FFM_ATTRS)),
                       (modules.CABiNetOutput, (self._pack_head, self.HEAD_ATTRS))):
            if isinstance(model, cls):
                standalone = v
                break
        self.block = isinstance(model, modules.ContextAggregationBlock)
        self.backbone = isinstance(model, modules.MobileNetV3)
        self.n_classes = model.n_classes if standalone is None else 0
        self.stamp = None
        self.launches = 0  # kernels enqueued by the last forward
        self.use_tc = precision == "bf16"
        self.debug = False
        self.stages = {}
        self.trace, self.trace_filter = None, None
        self.fuse_mbconv = True     # expand + depthwise (+ project) in one kernel (blocks whose tiles fit the shared memory)
        self.se_from_sums = True    # stride-1 SE blocks: gate from sums of the expanded activation, whole block in one kernel
        self.use_stem2 = True       # stems without the im2col tile (cabinet_stem_tc2)
        self.use_stem3 = True       # standalone backbone: its stem on the tensor cores (cabinet_stem3_tc), not conv2d_simt
        self.t_small_s2 = False     # stride-2 blocks with <= 64 expanded channels (Large f2) through cabinet_mbconv_t too
        self.t_k5s2 = True          # k5 stride-2 SE blocks (Large f4, f13) through cabinet_mbconv_t as well
        self.use_mbconv_t = True    # ... in the channel-major formulation (cabinet_mbconv_t) where it supports the block
        self.fold_se_relu = True    # ReLU SE blocks: gate folded into per-image project weights (relu(s*d) = s*relu(d))
        self.fold_ffm = True        # FFM gate folded into per-image head-conv weights (no rewrite of the fused feature map)
        # convb + x4 upsample + the low half of ffm.convblk as a 1/32-resolution conv + upsample-add in the convblk epilogue
        # (cabinet_conv_tc_up).  Correct and parity-tested, but measured SLOWER (convblk 72 -> 146 us): every output
        # element gathers 4 fp32 taps, 8x the bytes it writes, through a small L1 -> off by default
        self.fold_low_up = False
        # layers that walk their tiles back to front: their input (> L2) was written by the previous kernel, whose tail
        # is still L2 resident; the next layer then finds THIS layer's head in L2
        self.reverse_layers = frozenset()
        self.fuse_se = False        # SE apply as A-operand prologue of the project GEMM for every hard-swish SE block
        # ... or only for the blocks where it measured faster than scale_act + plain GEMM (tools/trace_se.py)
        self.fuse_se_blocks = frozenset({"mobile.f12", "mobile.f13"})
        self.use_cuda_graph = False
        self.sub_batch = 0          # > 0: run the schedule over chunks of this many images
        self._graphs = {}
        self._pool = None
        self._graph_seen = {}
        self.dual_stream = False    # experimental: two half-batches on two streams
        self._side = None
        self._scratch = []
        self.branch_overlap = True  # independent chains of the attention branch on side streams (fork / join by events)
        self._branch_streams, self._branch_events = [], {}
        self.sb_overlap = False     # experiment: spatial branch beside the backbone
        if packed is not None and standalone is not None:
            raise ValueError("packed weights exist for CABiNet engines only")
        if packed is not None:  # cached fold + pack of exactly these weights (checkpoint.load_packed verified the digest)
            missing = [a for a in self.PACKED_ATTRS if a not in packed]
            if missing:
                raise ValueError(f"packed weights lack {missing}")
            for a in self.PACKED_ATTRS:
                setattr(self, a, _from_plain(packed[a]))
            self.gamma = model.ab.a2block.gamma.detach().float().contiguous()
        else:
            with torch.no_grad():
                pack, attrs = standalone if standalone is not None else (self._pack, self.PACKED_ATTRS)
                pack(model)  # on the host ...
                for a in attrs:  # ... then one upload per packed tensor
                    setattr(self, a, _map_tensors(getattr(self, a), lambda t: t.to(self.dev)))

    def packed_state(self) -> dict:
        """Everything ``_pack`` produced as plain containers (dict / list / tuple / tensor / scalar / str): the cache
        file holds no pickled classes and loads with ``torch.load(weights_only=True)``."""
        return {a: _to_plain(getattr(self, a)) for a in self.PACKED_ATTRS}

    # ------------------------------------------------------------------ packing
    def _pack(self, m):
        wd = self.tdt
        mob = m.mobile
        self._pack_backbone(mob)

        sb = m.sb
        self.stem_tc = self.stem_tc2 = None
        if self.precision == "bf16":
            # fused stems: [80][192] bf16, k = (c*7 + ky)*8 + kx; the 3x3 stem sits in the centre of a 7x7 footprint
            w7, b7 = _fold(sb.conv1.conv.weight, None, sb.conv1.bn)
            w3, b3 = _fold(mob.features[0][0].weight, None, mob.features[0][1])
            pk = torch.zeros((80, 3, 7, 8), dtype=torch.float32, device=w7.device)
            pk[:64, :, :, 1:8] = w7  # kx = 0 is the zero-weight alignment slot
            pk[64:, :, 2:5, 3:6] = w3
            self.stem_tc = (pk.reshape(80, 168).contiguous(), torch.cat([b7, b3]).contiguous())
            wk = torch.zeros((80, 192), dtype=torch.float32, device=w7.device)
            wk[:, :168] = self.stem_tc[0]
            bias = self.stem_tc[1]
            b_hi = bias.to(torch.bfloat16).float()
            wk[:, 168], wk[:, 169] = b_hi, bias - b_hi  # bias rides in two spare K slots (A feeds 1.0 there)
            self.stem_tc = (wk.to(torch.bfloat16).contiguous(), bias)
            self.stem_tc2 = _stem_tc2_pack(pk, bias, b_hi)
        self._pack_sb(sb)
        ab = m.ab
        self._pack_ab(ab)
        ffm = m.ffm
        self._pack_ffm(ffm)
        # A 1x1 conv commutes with bilinear interpolation: convblk(cat[sb, up(low)]) = W_sb sb + up(W_low low) + b, and
        # low = convb(feat) is itself a 1x1 conv -> one 256 -> 256 conv at 1/32 resolution (W_low W_convb, bias
        # W_low b_convb) whose fp32 output the convblk epilogue upsamples and adds (cabinet_conv_tc_up).  The x4-upsampled
        # 256-channel tensor is never written and convblk's K shrinks from 384 to 128.
        self.ffm_sb = self.low_fold = None
        if self.precision == "bf16" and ffm.convblk.conv.kernel_size == (1, 1) and ab.convb.kernel_size == (1, 1):
            wf, bf_ = _fold(ffm.convblk.conv.weight, ffm.convblk.conv.bias, ffm.convblk.bn)
            n_sb = sb.conv_out.conv.out_channels
            w_low = wf[:, n_sb:, 0, 0].double()
            wb, bb = _fold(ab.convb.weight, ab.convb.bias, None)
            self.ffm_sb = ConvLayer(None, None, ACT_RELU, wd, "ffm.convblk", folded=(wf[:, :n_sb].contiguous(), bf_, 1, 0))
            self.low_fold = ConvLayer(None, None, ACT_NONE, wd, "ab.convb*ffm.low",
                                      folded=((w_low @ wb[:, :, 0, 0].double()).float()[:, :, None, None].contiguous(),
                                              (w_low @ bb.double()).float(), 1, 0))
        self._pack_head(m.conv_out)

    def _pack_sb(self, sb):
        """The SpatialBranch's four ConvBNReLU layers (reference: cabinet.py:108-129), BN folded."""
        wd = self.tdt
        self.sb1 = ConvLayer(sb.conv1.conv, sb.conv1.bn, ACT_RELU, torch.float32, "sb.conv1")  # reads the fp32 NCHW input
        self.sb2 = ConvLayer(sb.conv2.conv, sb.conv2.bn, ACT_RELU, wd, "sb.conv2")
        self.sb3 = ConvLayer(sb.conv3.conv, sb.conv3.bn, ACT_RELU, wd, "sb.conv3")
        self.sb4 = ConvLayer(sb.conv_out.conv, sb.conv_out.bn, ACT_RELU, wd, "sb.conv_out")

    def _pack_spatial(self, sb):
        """A standalone SpatialBranch: its layers + the weights of the sb.conv1-only tensor-core stem."""
        self._pack_sb(sb)
        self.stem_tc7 = None
        if self.precision == "bf16":
            # cabinet_stem7_tc: rows 0..63 of the cabinet_stem_tc2 pack (kx = 0 is the zero-weight alignment slot)
            w7, b7 = _fold(sb.conv1.conv.weight, None, sb.conv1.bn)
            pk = torch.zeros((64, 3, 7, 8), dtype=torch.float32, device=w7.device)
            pk[:, :, :, 1:8] = w7
            self.stem_tc7 = _stem_tc2_pack(pk, b7, b7.to(torch.bfloat16).float())

    def _pack_ab(self, ab):
        """The AttentionBranch (reference: cabinet.py:54-94), BN folded; b2 is b1's BatchNorm."""
        wd = self.tdt
        self.conva = ConvLayer(ab.conva[0], ab.conva[1], ACT_RELU, wd, "ab.conva")
        self._pack_cab(ab.a2block)
        self.convb = ConvLayer(ab.convb, None, ACT_NONE, wd, "ab.convb")
        self.b1 = ConvLayer(ab.b1, ab.b2, ACT_RELU, wd, "ab.b1")
        self.b4 = ConvLayer(ab.b4, None, ACT_NONE, wd, "ab.b4")

    def _pack_ffm(self, ffm):
        """The FeatureFusionModule's convblk and its channel gate (reference: cabinet.py:132-153), BN folded."""
        self.ffm_blk = ConvLayer(ffm.convblk.conv, ffm.convblk.bn, ACT_RELU, self.tdt, "ffm.convblk")
        self.ffm_gate = GateLayer(ffm.conv1.weight, None, ffm.conv2.weight, None, ACT_SIGMOID)

    def _pack_head(self, head):
        """CABiNetOutput (reference: cabinet.py:156-172), BN folded."""
        self.head_conv = ConvLayer(head.conv.conv, head.conv.bn, ACT_RELU, self.tdt, "conv_out.conv")
        self.head_out = ConvLayer(head.conv_out, None, ACT_NONE, self.tdt, "conv_out.conv_out")

    def _pack_backbone(self, mob):
        """The MobileNetV3's stem, blocks and last conv (reference: mobilenetv3.py:86-159,173-205), BN folded."""
        wd = self.tdt
        f32 = torch.float32
        # stems read the fp32 NCHW input directly; their (tiny) weights stay fp32
        self.stem = ConvLayer(mob.features[0][0], mob.features[0][1], ACT_HSWISH, f32, "mobile.stem")
        self.blocks = []
        for bi, blk in enumerate(list(mob.features)[1:], 1):
            s, c = blk.spec, blk.conv
            act = ACT_HSWISH if s["hs"] else ACT_RELU
            e = dict(spec=s, act=act)
            if s["expand"]:
                e["pw1"] = ConvLayer(c[0], c[1], act, wd, f"mobile.f{bi}.expand")
                e["dw"] = DwLayer(c[3], c[4], ACT_NONE if s["se"] else act, f"mobile.f{bi}.dw")
                se, pw2, bn2 = c[5], c[7], c[8]
                if self.precision == "bf16":
                    # fused-block side table: fp32 [chunks][k*k + 2][64] = depthwise taps, expand bias, depthwise bias
                    dwl, kk, nc = e["dw"], e["dw"].k ** 2, -(-e["dw"].c // 64)
                    aux = torch.zeros((nc * 64, kk + 2), dtype=f32, device=dwl.w.device)
                    aux[: dwl.c, :kk] = dwl.w.t()
                    aux[: dwl.c, kk + 1] = dwl.b
                    e["aux"] = aux.view(nc, 64, kk + 2).permute(0, 2, 1).contiguous()
                    p1 = e["pw1"]
                    if p1.cin % 8 == 0 and p1.cin % 64 <= 56 and p1.cin <= 248:
                        # expand weights with the bias as two extra K columns (bf16 hi + lo; the kernel feeds 1.0 there);
                        # K = Cin + 2 padded to whole 64-channel K blocks
                        wb = torch.zeros((-(-p1.cout // 16) * 16, (p1.cin // 64 + 1) * 64), dtype=f32, device=dwl.w.device)
                        wb[: p1.cout, : p1.cin] = p1.tc[: p1.cout, 0, : p1.cin].float()
                        hi = p1.b.to(torch.bfloat16).float()
                        wb[: p1.cout, p1.cin], wb[: p1.cout, p1.cin + 1] = hi, p1.b - hi
                        e["w1b"] = wb.to(torch.bfloat16).contiguous()
                        # channel-major kernel (cabinet_mbconv_t): chunks of 128 TMEM lanes; widths <= 64 are replicated
                        # twice along the lanes.  Same columns as w1b; taps + depthwise bias in the same row order.
                        ch = 64 if dwl.c <= 64 else 128
                        nct = 1 if dwl.c <= 64 else -(-dwl.c // 128)
                        flat = torch.zeros((nct * ch, wb.shape[1]), dtype=f32, device=dwl.w.device)
                        flat[: dwl.c] = wb[: dwl.c]
                        e["w1t"] = (flat.view(nct, ch, -1).repeat(1, 128 // ch, 1).reshape(nct * 128, -1)
                                    .to(torch.bfloat16).contiguous())
                        fa = torch.zeros((nct * ch, kk + 1), dtype=f32, device=dwl.w.device)
                        fa[: dwl.c, :kk] = dwl.w.t()
                        fa[: dwl.c, kk] = dwl.b
                        e["auxt"] = fa.view(nct, ch, kk + 1).repeat(1, 128 // ch, 1).permute(0, 2, 1).contiguous()
            else:
                e["dw"] = DwLayer(c[0], c[1], act, f"mobile.f{bi}.dw")
                se, pw2, bn2 = c[3], c[4], c[5]
            if s["se"]:
                e["se"] = GateLayer(se.fc[0].weight, se.fc[0].bias, se.fc[2].weight, se.fc[2].bias, ACT_HSIGMOID)
            e["pw2"] = ConvLayer(pw2, bn2, ACT_NONE, wd, f"mobile.f{bi}.project")
            if (not s["expand"] and not s["se"] and s["identity"] and s["k"] == 3 and s["exp"] in (8, 16, 32)
                    and self.precision == "bf16"):
                w2, b2 = _fold(pw2.weight, pw2.bias, bn2)  # fused whole-block kernel keeps the pointwise in fp32
                e["fused_pw"] = (w2.reshape(w2.shape[0], -1).contiguous(), b2.contiguous())
            self.blocks.append(e)
        self.last = ConvLayer(mob.conv[0], mob.conv[1], ACT_HSWISH, wd, "mobile.conv")

    def _pack_mobilenet(self, mob):
        """A standalone MobileNetV3: the backbone's layers + the weights of the backbone-only tensor-core stem."""
        self._pack_backbone(mob)
        self.stem_tc3 = None
        if self.precision == "bf16":
            # cabinet_stem3_tc: W[o][ky][s][c], slot s = kx + 1 (slot 0: no tap; its constant-1 channel c = 3 carries
            # the bias, hi part at ky 1, lo part at ky 0) as UMMA core matrices [ky][k chunk][o][8]
            w3, b3 = _fold(mob.features[0][0].weight, None, mob.features[0][1])
            wn = torch.zeros((16, 3, 4, 4), dtype=torch.float32, device=w3.device)
            wn[:, :, 1:, :3] = w3.permute(0, 2, 3, 1)
            b_hi = b3.to(torch.bfloat16).float()
            wn[:, 1, 0, 3], wn[:, 0, 0, 3] = b_hi, b3 - b_hi
            self.stem_tc3 = wn.view(16, 3, 2, 8).permute(1, 2, 0, 3).contiguous().to(torch.bfloat16)

    def _pack_cab(self, cab):
        """The ContextAggregationBlock's layers (reference: cab.py:84-129,170-184,192-216), BN folded."""
        wd = self.tdt
        ga = cab.global_attn
        self.to_q = ConvLayer(ga.to_query[0], ga.to_query[1], ACT_RELU, wd, "cab.to_query")
        self.to_k = ConvLayer(ga.to_key[0], ga.to_key[1], ACT_RELU, wd, "cab.to_key")
        self.to_v = ConvLayer(ga.to_value, None, ACT_NONE, wd, "cab.to_value")
        self.psp_k = ConvLayer(ga.psp_key.project, None, ACT_NONE, wd, "cab.psp_key")
        self.psp_v = ConvLayer(ga.psp_value.project, None, ACT_NONE, wd, "cab.psp_value")
        self.proj_out = ConvLayer(ga.project_out, None, ACT_NONE, wd, "cab.project_out")
        self.local = [DwLayer(d.block[0], d.block[1], ACT_RELU, f"cab.local{i}")
                      for i, d in enumerate(cab.local_attn.refine)]
        self.gamma = _host(cab.gamma).contiguous()
        self.key_ch = self.to_k.cout
        # to_query | to_key | to_value read the same tensor: one 256 -> 3 x 128 GEMM, ReLU on the first 2 x 128 outputs
        self.qkv = None
        if (self.precision == "bf16" and all(L.tc is not None and L.kh == 1 for L in (self.to_q, self.to_k, self.to_v))
                and self.to_q.cout == self.to_k.cout == self.to_v.cout and self.to_q.cout % 16 == 0):
            self.qkv = (torch.cat([L.tc[: L.cout] for L in (self.to_q, self.to_k, self.to_v)], 0).contiguous(),
                        torch.cat([self.to_q.b, self.to_k.b, self.to_v.b]).contiguous())

    # ------------------------------------------------------------------ kernel wrappers
    @property
    def stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def _run(self, kernel: str, layer: str, nbytes: int, flops: int, fn, *args):
        """Enqueue one kernel.  With tracing on, bracket it with CUDA events on the launching stream and keep
        its ALGORITHMIC bytes/flops (each operand once, SURVEY 8d) for the roofline report.  ``nbytes`` may be a pair
        (per-layer-fusion model bytes of SURVEY 8d, bytes the block-fused kernel itself has to move)."""
        nbytes, fused_bytes = nbytes if isinstance(nbytes, tuple) else (nbytes, nbytes)
        tr = self.trace
        if tr is not None and (self.trace_filter is None or kernel in self.trace_filter):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*args)
            e1.record()
            tr.append((kernel, layer, nbytes, flops, e0, e1, fused_bytes))
        else:
            rc = fn(*args)
        check(rc, f"{kernel}[{layer}]")
        self.launches += 1

    def new(self, N, H, W, C, dtype=None) -> Map:
        t = torch.empty((N, H, W, C), dtype=dtype or self.tdt, device=self.dev)
        return Map(t, N, H, W, C, C)

    def conv(self, x: Map, L: ConvLayer, out: Optional[Map] = None, res: Optional[Map] = None, out_dtype=None,
             nchw_input: Optional[torch.Tensor] = None, a_scale: Optional[torch.Tensor] = None, a_act: int = 0) -> Map:
        """Dense conv + bias + act (+ residual).  ``nchw_input``: read the fp32 NCHW network input in place."""
        if nchw_input is not None:
            N, _, H, W = nchw_input.shape
            xptr, xdt, xes = nchw_input.data_ptr(), F32, 4
            sxn, sxh, sxw, sxc = 3 * H * W, W, 1, H * W
            cin = 3
        else:
            N, H, W, cin = x.N, x.H, x.W, x.C
            xptr, xdt, xes = x.ptr, x.dt, x.t.element_size()
            sxn, sxh, sxw, sxc = H * W * x.ld, W * x.ld, x.ld, 1
        assert cin == L.cin, (L.name, cin, L.cin)
        OH, OW = _out_size(H, L.kh, L.stride, L.pad), _out_size(W, L.kw, L.stride, L.pad)
        if out is None:
            out = self.new(N, OH, OW, L.cout, out_dtype)
        assert (out.N, out.H, out.W, out.C) == (N, OH, OW, L.cout), L.name
        M = N * OH * OW
        nbytes = (N * H * W * cin * xes + M * L.cout * out.t.element_size() + L.w.numel() * L.w.element_size()
                  + (M * L.cout * res.t.element_size() if res is not None else 0))
        flops = 2 * M * L.cout * L.cin * L.kh * L.kw
        if (self.use_tc and L.tc is not None and nchw_input is None and x.dt == BF16 and x.ld % 8 == 0
                and x.off % 8 == 0 and (L.stride == 1 or (H >= 2 and W >= 2))
                and (out.dt == F32 or (out.ld % 8 == 0 and out.off % 8 == 0))):
            self._conv_tc(x, L, out, res, OH, OW, nbytes, flops, a_scale, a_act)
            return out
        assert a_scale is None, "the SE prologue exists on the tcgen05 path only"
        wdt = BF16 if L.w.dtype == torch.bfloat16 else F32
        self._run("conv2d_simt", L.name, nbytes, flops, self.lib.cabinet_conv2d_simt,
                  xptr, xdt, sxn, sxh, sxw, sxc, 0, L.w.data_ptr(), wdt, L.w.shape[1], 1, 0, L.b.data_ptr(),
                  res.ptr if res is not None else None, res.ld if res is not None else 0,
                  out.ptr, out.dt, out.ld, 0, 1, N, H, W, cin, L.cout, L.kh, L.kw, L.stride, L.pad, OH, OW, L.act,
                  1.0, self.stream)
        return out

    REVERSE_TILES = 0x100  # CABINET_CONV_REVERSE_TILES

    def _conv_tc(self, x: Map, L: ConvLayer, out: Map, res: Optional[Map], OH, OW, nbytes, flops, a_scale=None, a_act=0):
        self._run("conv_tc", L.name, nbytes, flops, self.lib.cabinet_conv_tc_se, x.ptr, x.ld, x.N, x.H, x.W, x.C,
                  a_scale.data_ptr() if a_scale is not None else None, a_act,
                  L.tc.data_ptr(), L.cout, L.kh, L.kw, L.stride, L.pad, L.b.data_ptr(),
                  res.ptr if res is not None else None, res.ld if res is not None else 0, out.ptr, out.dt, out.ld,
                  OH, OW, L.act | (self.REVERSE_TILES if L.name in self.reverse_layers else 0), self.stream)

    def dwconv(self, x: Map, L: DwLayer, gap: Optional[torch.Tensor] = None):
        """Depthwise conv + bias + act.  ``gap`` ([N, C], zeroed): also the per-(image, channel) sums of the written
        values, deterministic.  bf16 path: int64 fixed-point accumulators (``cabinet_gate_fc(in_fixed=1)`` consumes
        them); fp32 parity path: fp32 sums by the two-level ``channel_sum`` over the written tensor.
        -> (out, gap_is_fixed_point)"""
        p = (L.k - 1) // 2
        OH, OW = _out_size(x.H, L.k, L.stride, p), _out_size(x.W, L.k, L.stride, p)
        out = self.new(x.N, OH, OW, x.C)
        es = x.t.element_size()
        nbytes = x.N * x.C * (x.H * x.W + OH * OW) * es + L.w.numel() * 4
        flops = 2 * x.N * OH * OW * x.C * L.k * L.k
        if self.use_tc and x.dt == BF16 and x.ld % 8 == 0 and x.off % 8 == 0:
            self._run("dwconv_tma", L.name, nbytes, flops, self.lib.cabinet_dwconv_tma, x.ptr, x.ld, L.w.data_ptr(),
                      L.b.data_ptr(), out.ptr, out.ld, x.N, x.H, x.W, x.C, L.k, L.stride, OH, OW,
                      L.act | (self.REVERSE_TILES if L.name in self.reverse_layers else 0),
                      gap.data_ptr() if gap is not None else None, self.stream)
            return out, True
        self._run("dwconv", L.name, nbytes, flops, self.lib.cabinet_dwconv, x.ptr, x.ld, L.w.data_ptr(),
                  L.b.data_ptr(), out.ptr, out.ld, x.dt, x.N, x.H, x.W, x.C, L.k, L.stride, OH, OW, L.act, None,
                  self.stream)
        if gap is not None:  # parity mode: the deterministic two-level channel sum over the written tensor
            self.channel_sum(out, gap, L.name)
        return out, False

    def channel_sum(self, x: Map, out: torch.Tensor, name: str, scratch: Optional[torch.Tensor] = None):
        """out[n][c] = sum over pixels of x (deterministic: per-block partials, fixed-order final sum)."""
        if scratch is None:
            scratch = torch.zeros(128 + x.N * 64 * x.C, dtype=torch.float32, device=self.dev)
            self.launches += 1
        self._run("channel_sum", name, 0, 0, self.lib.cabinet_channel_sum, x.ptr, x.ld, x.dt, x.N, x.H * x.W, x.C,
                  out.data_ptr(), scratch.data_ptr(), scratch.numel() * 4, self.stream)

    # ------------------------------------------------------------------ independent branches on side streams
    class _Branch:
        """Kernels enqueued inside the block go to side stream `i` (forked from the current stream); `joined(t)` marks a
        tensor that the main stream consumes after `_join(i)`.  The small kernels of the attention branch are latency
        bound, so two independent chains side by side cost the longer one, not the sum.  Works eagerly and under CUDA
        graph capture (fork / join by events)."""

        def __init__(self, eng, i):
            self.eng, self.i = eng, i

        def __enter__(self):
            eng = self.eng
            if not eng.branch_overlap or eng.trace is not None or torch.device(eng.dev).type != "cuda":
                self.ctx = None
                return lambda t: None
            self.main = torch.cuda.current_stream(eng.dev)
            while len(eng._branch_streams) <= self.i:
                eng._branch_streams.append(torch.cuda.Stream(eng.dev))
            side = eng._branch_streams[self.i]
            ev = torch.cuda.Event()
            ev.record(self.main)
            side.wait_event(ev)
            self.ctx = torch.cuda.stream(side)
            self.ctx.__enter__()
            return lambda t: t.record_stream(self.main)

        def __exit__(self, *a):
            if self.ctx is not None:
                eng = self.eng
                ev = torch.cuda.Event()
                ev.record(eng._branch_streams[self.i])
                eng._branch_events[self.i] = ev
                self.ctx.__exit__(*a)
            return False

    def _branch(self, i):
        return Engine._Branch(self, i)

    def _join(self, i):
        ev = self._branch_events.pop(i, None)
        if ev is not None:
            torch.cuda.current_stream(self.dev).wait_event(ev)

    def mbconv_fused(self, x: Map, e: dict, gap: Optional[torch.Tensor], act_dw: Optional[int] = None,
                     se_scale: Optional[torch.Tensor] = None) -> Map:
        """Inverted-residual block with the expanded activation kept on chip (reference: mobilenetv3.py:126-159).
        ``gap`` given (SE blocks; [N, Cexp] int64 fixed point, zeroed): returns the pre-SE depthwise output and
        accumulates its pooling sums; else the block output (project + identity included)."""
        s, pw1, dw, pw2 = e["spec"], e["pw1"], e["dw"], e["pw2"]
        pad = (dw.k - 1) // 2
        OH, OW = _out_size(x.H, dw.k, dw.stride, pad), _out_size(x.W, dw.k, dw.stride, pad)
        project = gap is None
        assert se_scale is None or project
        cy = pw2.cout if project else dw.c
        out = self.new(x.N, OH, OW, cy)
        nbytes = (x.N * x.H * x.W * x.C + x.N * OH * OW * cy) * 2 + pw1.w.numel() * 2 + dw.w.numel() * 4
        flops = 2 * x.N * x.H * x.W * x.C * dw.c + 2 * x.N * OH * OW * dw.c * dw.k * dw.k
        # SURVEY 8(d)'s per-layer-fusion model: the expand conv writes / the depthwise conv reads the expanded tensor, the
        # depthwise conv writes / the project conv reads its output -- traffic this kernel keeps on chip
        model = nbytes + 2 * x.N * x.H * x.W * dw.c * 2 + (2 * x.N * OH * OW * dw.c * 2 if project else 0)
        if project:
            extra = pw2.w.numel() * 2 + (x.N * OH * OW * cy * 2 if s["identity"] else 0)
            nbytes += extra
            model += extra
            flops += 2 * x.N * OH * OW * dw.c * pw2.cout
        nbytes = (model, nbytes)
        # (stride-2 blocks with <= 64 expanded channels -- Large f2 -- have 32-pixel tiles with four outputs per thread
        # there: latency bound, 0.33 ms against 0.18 ms for the pixel-major kernel)
        use_t = (self.use_mbconv_t and "w1t" in e and not e.get("no_t")
                 and not (dw.stride == 2 and dw.c <= 64 and not self.t_small_s2)
                 and (not project or (pw2.cout <= 128 and pw2.cout % 8 == 0 and (dw.k == 3 or dw.stride == 1))))
        if use_t:
            try:
                self._run("mbconv_t", dw.name.replace(".dw", "") + ("" if project else ".expand+dw"), nbytes, flops,
                          self.lib.cabinet_mbconv_t, x.ptr, x.ld, x.N, x.H, x.W, x.C, e["w1t"].data_ptr(),
                          e["auxt"].data_ptr(), dw.c, pw1.act, dw.k, dw.stride, dw.act if act_dw is None else act_dw,
                          pw2.tc.data_ptr() if project else None, pw2.b.data_ptr() if project else None,
                          pw2.cout if project else 0, 1 if project and s["identity"] else 0, out.ptr, out.ld, OH, OW,
                          gap.data_ptr() if gap is not None else None,
                          se_scale.data_ptr() if se_scale is not None else None, self.stream)
                return out
            except ValueError as err:  # outside the kernel's shared-memory / TMEM budget: the pixel-major kernel
                if "budget" not in str(err):
                    raise
                e["no_t"] = True
        if se_scale is not None:
            raise ValueError("budget: the squeeze-excite gate input exists in cabinet_mbconv_t only")
        self._run("mbconv_fused", dw.name.replace(".dw", "") + ("" if project else ".expand+dw"), nbytes, flops,
                  self.lib.cabinet_mbconv_fused, x.ptr, x.ld, x.N, x.H, x.W, x.C, e["w1b"].data_ptr(), e["aux"].data_ptr(),
                  dw.c, pw1.act, dw.k, dw.stride, dw.act if act_dw is None else act_dw,
                  pw2.tc.data_ptr() if project else None, pw2.b.data_ptr() if project else None,
                  pw2.cout if project else 0, 1 if project and s["identity"] else 0, out.ptr, out.ld, OH, OW,
                  gap.data_ptr() if gap is not None else None, self.stream)
        return out

    def _se_from_sums_ok(self, x: Map, e: dict) -> bool:
        s, dw, pw2 = e["spec"], e["dw"], e["pw2"]
        p = (dw.k - 1) // 2
        if isinstance(self.se_from_sums, (set, frozenset)) and dw.name[:-3] not in self.se_from_sums:
            return False
        elif self.se_from_sums is True and dw.k != 3:
            return False  # k5: the 8 x 8-tile project kernel + the sums pass measured no faster than the three-kernel path
        return (self.use_mbconv_t and not self.debug and not e.get("no_sums") and not e.get("no_t") and "w1t" in e
                and s["s"] == 1 and dw.c > 64 and 2 * p <= min(x.H, x.W) and max(x.H, x.W) <= 256
                and pw2.tc is not None and pw2.cout <= 128 and pw2.cout % 8 == 0)

    def se_block_one_kernel(self, x: Map, e: dict, gap: torch.Tensor) -> Map:
        """expand_sums -> gate layers -> mbconv_t(se_scale): reference mobilenetv3.py:126-159 with SELayer :68-83.
        ``gap``: this block's zeroed [N, Cexp] int64 fixed-point pooling accumulator."""
        dw, pw1 = e["dw"], e["pw1"]
        N = x.N
        nsplit = 0  # automatic: about two (image, part) units per persistent CTA
        name = dw.name.replace(".dw", "")
        self._run("expand_sums", name + ".sums", N * x.H * x.W * x.C * 2, 2 * N * x.H * x.W * x.C * dw.c,
                  self.lib.cabinet_expand_sums, x.ptr, x.ld, N, x.H, x.W, x.C, e["w1t"].data_ptr(), e["auxt"].data_ptr(),
                  dw.c, pw1.act, dw.k, nsplit, gap.data_ptr(), self.stream)
        scale = self.gate(gap.view(N, -1), x.H * x.W, e["se"], dw.name, True)
        # expand form: SE on the BN output, then the activation (F10)
        return self.mbconv_fused(x, e, None, act_dw=e["act"], se_scale=scale)

    def gate(self, gap: torch.Tensor, hw: int, G: GateLayer, name: str, fixed: bool = False) -> torch.Tensor:
        """Channel gate of SE / FFM: two batched tiny FC layers (mean -> ReLU hidden -> gate), fp32.  ``fixed``:
        ``gap`` holds int64 fixed-point sums (the depthwise kernels' deterministic pooling accumulators)."""
        n = gap.shape[0]
        hidden = torch.empty((n, G.cmid), dtype=torch.float32, device=self.dev)
        scale = torch.empty((n, G.c), dtype=torch.float32, device=self.dev)
        self._run("gate_fc", name, G.w1.numel() * 4, 2 * n * G.c * G.cmid, self.lib.cabinet_gate_fc, gap.data_ptr(),
                  1.0 / hw, G.w1.data_ptr(), G.b1.data_ptr() if G.b1 is not None else None, hidden.data_ptr(), n, G.c,
                  G.cmid, ACT_RELU, int(fixed), self.stream)
        self._run("gate_fc", name, G.w2.numel() * 4, 2 * n * G.c * G.cmid, self.lib.cabinet_gate_fc, hidden.data_ptr(),
                  1.0, G.w2.data_ptr(), G.b2.data_ptr() if G.b2 is not None else None, scale.data_ptr(), n, G.cmid,
                  G.c, G.gate, 0, self.stream)
        return scale

    def gate_scale_weights(self, gap: torch.Tensor, fixed: bool, hw: int, G: GateLayer, w_tc: torch.Tensor, wimg: torch.Tensor,
                           cin: int, plus_one: bool, name: str):
        """Gate MLP + per-image copies of a conv_tc weight pack scaled by (gate + plus_one), one launch."""
        n = wimg.shape[0]
        self._run("gate_scale_weights", name, wimg.numel() * 2 + (G.w1.numel() + G.w2.numel()) * 4, 4 * n * G.c * G.cmid,
                  self.lib.cabinet_gate_scale_weights, gap.data_ptr(), int(fixed), 1.0 / hw, G.w1.data_ptr(),
                  G.b1.data_ptr() if G.b1 is not None else None, G.w2.data_ptr(),
                  G.b2.data_ptr() if G.b2 is not None else None, G.gate, G.c, G.cmid, w_tc.data_ptr(), wimg.data_ptr(), n,
                  w_tc.shape[0], w_tc.shape[1], w_tc.shape[2], int(plus_one), self.stream)

    def scale_act(self, x: Map, scale: torch.Tensor, act: int, name: str, plus_one: bool = False):
        # not in the per-layer-fusion byte model (SE scale / FFM gate are "free riders" there): counted as 0 algorithmic
        self._run("scale_act", name, 0, 0, self.lib.cabinet_scale_act, x.ptr, x.ld, x.dt, scale.data_ptr(), x.N,
                  x.H * x.W, x.C, act, int(plus_one), self.stream)

    def psp(self, x: Map, L: ConvLayer) -> Map:
        """PSP encoder: pools -> 5C concat -> 1x1 project (reference: cab.py:65-76)."""
        pooled = torch.empty((x.N, 110, x.C), dtype=torch.float32, device=self.dev)
        es = x.t.element_size()
        need = 128 + x.N * (110 + 256 * x.C)
        if self._scratch and self._scratch[-1].numel() >= need:
            scratch = self._scratch.pop()  # zeroed with the per-forward memset (tickets must start at zero)
        else:
            scratch = torch.zeros(need, dtype=torch.float32, device=self.dev)
            self.launches += 1
        self._run("psp_pool", L.name, x.N * x.H * x.W * x.C * es, 0, self.lib.cabinet_psp_pool, x.ptr, x.ld, x.dt,
                  pooled.data_ptr(), x.N, x.H, x.W, x.C, scratch.data_ptr(), scratch.numel() * 4, self.stream)
        cat = self.new(x.N, x.H, x.W, 5 * x.C)
        self._run("psp_concat", L.name, 0, 0, self.lib.cabinet_psp_concat, x.ptr, x.ld, pooled.data_ptr(), cat.ptr,
                  cat.ld, x.dt, x.N, x.H, x.W, x.C, self.stream)
        return self.conv(cat, L)

    def attention(self, q: Map, k: Map, v: Map) -> Map:
        """softmax(q k^T / sqrt(dk)) v per image (reference: cab.py:149-153).  q, k: [N, L, dk], v: [N, L, dv] dense;
        -> ctx [N, L, dv].  The tensor-core kernel takes dk in {64, 128, 256} x dv in {64, 128} (bf16, 16-byte rows);
        every other width / the fp32 parity mode runs the CUDA-core GEMMs + softmax."""
        N, Lq, d, dv = q.N, q.H * q.W, q.C, v.C
        es = q.t.element_size()
        ctx = self.new(q.N, q.H, q.W, dv)
        if (self.use_tc and d in (64, 128, 256) and dv in (64, 128) and q.dt == BF16
                and all(m.ld % 8 == 0 and m.off % 8 == 0 for m in (q, k, v))):
            vt = torch.empty((N, dv, -(-Lq // 8) * 8), dtype=torch.bfloat16, device=self.dev)
            nbytes, flops = 2 * N * Lq * (d + dv) * es, 2 * N * Lq * Lq * (d + dv)
            if d == dv == 128:  # CABiNet's attention: the original entry point
                self._run("attention_tc", "cab.attention", nbytes, flops, self.lib.cabinet_attention_tc, q.ptr, q.ld,
                          k.ptr, k.ld, v.ptr, v.ld, vt.data_ptr(), ctx.ptr, ctx.ld, N, Lq, d, float(d) ** -0.5, self.stream)
            else:
                self._run("attention_tc", "cab.attention", nbytes, flops, self.lib.cabinet_attention_tc_dkdv, q.ptr, q.ld,
                          k.ptr, k.ld, v.ptr, v.ld, vt.data_ptr(), ctx.ptr, ctx.ld, N, Lq, d, dv, float(d) ** -0.5,
                          self.stream)
            self.launches += 1  # the V transpose pre-kernel
            return ctx
        s = torch.empty((N, Lq, Lq), dtype=torch.float32, device=self.dev)
        # S[b][i][j] = alpha * sum_c q[b][i][c] k[b][j][c]   (k acts as the [Cout=L][K=dk] "weights")
        self._run("conv2d_simt", "cab.qk", 2 * N * Lq * d * es, 2 * N * Lq * Lq * d, self.lib.cabinet_conv2d_simt,
                  q.ptr, q.dt, 0, 0, q.ld, 1, Lq * q.ld, k.ptr, k.dt, k.ld, 1, Lq * k.ld, None, None, 0,
                  s.data_ptr(), F32, Lq, Lq * Lq, N, 1, 1, Lq, d, Lq, 1, 1, 1, 0, 1, Lq, ACT_NONE, float(d) ** -0.5,
                  self.stream)
        p = torch.empty((N, Lq, Lq), dtype=self.tdt, device=self.dev)
        self._run("softmax_rows", "cab.softmax", 0, 0, self.lib.cabinet_softmax_rows, s.data_ptr(), p.data_ptr(),
                  self.dt, N * Lq, Lq, self.stream)
        # ctx[b][i][c] = sum_j P[b][i][j] v[b][j][c]   (v read as [Cout=dv][K=L] with strides (1, ld))
        self._run("conv2d_simt", "cab.pv", 2 * N * Lq * dv * es, 2 * N * Lq * Lq * dv, self.lib.cabinet_conv2d_simt,
                  p.data_ptr(), self.dt, 0, 0, Lq, 1, Lq * Lq, v.ptr, v.dt, 1, v.ld, Lq * v.ld, None, None, 0,
                  ctx.ptr, ctx.dt, ctx.ld, Lq * ctx.ld, N, 1, 1, Lq, Lq, dv, 1, 1, 1, 0, 1, Lq, ACT_NONE, 1.0,
                  self.stream)
        return ctx

    def cab(self, feat: Map, out: Map):
        """ContextAggregationBlock: out = gamma * global(feat) + local(feat) (reference: cab.py:131-162,175-184,213-216).
        ``feat`` dense; ``out`` may be a channel slice of a wider buffer."""
        N, h, w = feat.N, feat.H, feat.W
        if self.qkv is not None and self.use_tc and feat.dt == BF16:
            kc = self.key_ch
            qkv = self.new(N, h, w, 3 * kc)
            M = N * h * w
            self._run("conv_tc", "cab.to_query|key|value", (M * (feat.C + 3 * kc) + self.qkv[0].numel()) * 2,
                      2 * M * 3 * kc * feat.C, self.lib.cabinet_conv_tc_split_act, feat.ptr, feat.ld, N, h, w, feat.C,
                      self.qkv[0].data_ptr(), 3 * kc, 1, 1, 1, 0, self.qkv[1].data_ptr(), qkv.ptr, qkv.dt, qkv.ld, h, w,
                      ACT_RELU, 2 * kc, self.stream)
            q = qkv.slice(0, kc)
            with self._branch(1) as joined:     # value PSP chain beside the key PSP chain
                v = self.psp(qkv.slice(2 * kc, kc), self.psp_v)
                joined(v.t)
            k = self.psp(qkv.slice(kc, kc), self.psp_k)
        else:
            q = self.conv(feat, self.to_q)
            k = self.psp(self.conv(feat, self.to_k), self.psp_k)
            v = self.psp(self.conv(feat, self.to_v), self.psp_v)
        with self._branch(0) as joined:         # local attention (three depthwise convs) beside the global attention
            r = feat
            for L in self.local:
                r, _ = self.dwconv(r, L)
            joined(r.t)
        self._join(1)
        ctx = self.attention(q, k, v)
        g = self.conv(ctx, self.proj_out)
        self._join(0)
        es = feat.t.element_size()
        self._run("cab_combine", "cab", 2 * N * h * w * feat.C * es, 0, self.lib.cabinet_cab_combine, g.ptr, feat.ptr,
                  r.ptr, out.ptr, out.ld, self.gamma.data_ptr(), self.dt, N * h * w, feat.C, self.stream)

    def relayout(self, src: torch.Tensor, src_strides, dst: torch.Tensor, dst_strides, N, H, W, C, name: str):
        """dst = src element for element, between two (N, H, W, C) stride patterns and any two float dtypes (NCHW <->
        NHWC at a standalone block's boundary): cabinet_resample_sep with identity row operators."""
        from .train_engine import _Tables

        if getattr(self, "_tables", None) is None:
            self._tables = _Tables(self.dev)
        if {src.dtype, dst.dtype} == {torch.bfloat16, torch.float16}:  # no kernel for this pair: through fp32
            tmp = torch.empty((N, H, W, C), dtype=torch.float32, device=self.dev)
            self.relayout(src, src_strides, tmp, (H * W * C, W * C, C, 1), N, H, W, C, name)
            src, src_strides = tmp, (H * W * C, W * C, C, 1)
        ty, tx = self._tables.get("identity", H, H, False), self._tables.get("identity", W, W, False)
        self._run("resample_sep", name, N * H * W * C * (src.element_size() + dst.element_size()), 0,
                  self.lib.cabinet_resample_sep, src.data_ptr(), dtype_code(src.dtype), *src_strides, dst.data_ptr(),
                  dtype_code(dst.dtype), *dst_strides, N, H, W, C, *(t.data_ptr() for t in ty), *(t.data_ptr() for t in tx),
                  0, self.stream)

    @torch.no_grad()
    def forward_block(self, x: torch.Tensor) -> torch.Tensor:
        """Standalone ContextAggregationBlock: (N, C, H, W) fp32 / bf16 / fp16 -> the same shape and dtype."""
        N, C, H, W = x.shape
        y = torch.empty_like(x, memory_format=torch.contiguous_format)
        self.launches = 0
        if N == 0 or H * W == 0:
            return y
        nchw = lambda t: (t.stride(0), t.stride(2), t.stride(3), t.stride(1))  # noqa: E731  (n, y, x, c) strides
        with self._guard():
            self._scratch = []  # the PSP pools take freshly zeroed scratch
            feat, out = self.new(N, H, W, C), self.new(N, H, W, C)
            self.relayout(x, nchw(x), feat.t, (H * W * C, W * C, C, 1), N, H, W, C, "cab.in")
            self.cab(feat, out)
            self.relayout(out.t, (H * W * C, W * C, C, 1), y, nchw(y), N, H, W, C, "cab.out")
        return y

    def mobilenet(self, f: Map, gap_all: torch.Tensor, out: Optional[Map] = None) -> Map:
        """The backbone after its stem: the inverted-residual blocks and ``mobile.conv`` (reference: mobilenetv3.py:
        102-159,202-205).  ``f``: the stem's output; ``gap_all``: zeroed [>= 2 x SE blocks][N * 1024] fp32 (the SE pooling
        sums); ``out``: where ``mobile.conv`` writes (a channel slice of CABiNet's b1 concat buffer) or None."""
        N, dev = f.N, self.dev
        gi = 0
        for e in self.blocks:
            s = e["spec"]
            if "fused_pw" in e and self.use_tc and f.ld % 8 == 0 and f.off % 8 == 0:
                o = self.new(f.N, f.H, f.W, s["out"])
                dw = e["dw"]
                es = f.t.element_size()
                self._run("mbconv_noexpand_fused", dw.name.replace(".dw", ""), 2 * f.N * f.H * f.W * f.C * es,
                          2 * f.N * f.H * f.W * f.C * (9 + f.C), self.lib.cabinet_mbconv_noexpand_fused, f.ptr, f.ld,
                          dw.w.data_ptr(), dw.b.data_ptr(), e["fused_pw"][0].data_ptr(), e["fused_pw"][1].data_ptr(),
                          o.ptr, o.ld, f.N, f.H, f.W, f.C, dw.act, self.stream)
                f = o
                continue
            fuse = (s["expand"] and self.fuse_mbconv and self.use_tc and f.dt == BF16 and f.ld % 8 == 0
                    and f.off % 8 == 0 and s["exp"] % 8 == 0 and ("se" in e or s["out"] <= 160) and "w1b" in e
                    and not e.get("nofuse")
                    # 5x5 stride-2 tiles are 4 x 8 outputs behind an 11 x 19 halo: the pixel-major kernel measured slower
                    # than expand + dwconv_tma there; the channel-major one takes SE blocks (depthwise-output mode)
                    and not (s["k"] == 5 and s["s"] == 2 and not (self.use_mbconv_t and self.t_k5s2 and "se" in e)))
            d = None
            gap_fixed = False
            if fuse and "se" in e and self.se_from_sums and self._se_from_sums_ok(f, e):
                # stride-1 squeeze-excite block: the gate from border-corrected sums of the expanded activation (its mean
                # after the depthwise conv is linear in them), then the WHOLE block as one kernel
                try:
                    f = self.se_block_one_kernel(f, e, gap_all[2 * gi:2 * gi + 2].view(-1)[: 2 * N * s["exp"]])
                    gi += 1
                    continue
                except ValueError as err:
                    if "budget" not in str(err):
                        raise
                    e["no_sums"] = True
            if fuse:
                # expand -> depthwise (-> project + identity): the expanded activation never leaves the SM
                gap = None
                if "se" in e:
                    gap, gap_fixed = gap_all[2 * gi:2 * gi + 2].view(-1)[: 2 * N * s["exp"]], True
                # ReLU SE blocks: relu(s * d) = s * relu(d) (s = hard-sigmoid >= 0), so the kernel applies the ReLU and the
                # gate is folded into per-image project weights -- no scale_act pass over the expanded tensor
                pw2l = e["pw2"]
                fold_se = ("se" in e and self.fold_se_relu and e["act"] == ACT_RELU and not self.debug
                           and pw2l.tc is not None and pw2l.kh == 1 and (f.H // s["s"]) * (f.W // s["s"]) % 128 == 0
                           and f.H % s["s"] == 0 and f.W % s["s"] == 0)
                try:
                    d = self.mbconv_fused(f, e, gap, ACT_RELU if fold_se else None)
                except ValueError as err:  # block shape outside the kernel's shared-memory / TMEM budget
                    if "budget" not in str(err):
                        raise
                    e["nofuse"], fuse = True, False
            if fuse and "se" not in e:
                f = d
                continue
            h = self.conv(f, e["pw1"]) if s["expand"] and not fuse else f
            if "se" in e:
                if not fuse:
                    gap = gap_all[2 * gi:2 * gi + 2].view(-1)[: 2 * N * s["exp"]]
                    d, gap_fixed = self.dwconv(h, e["dw"], gap)
                gi += 1
                if fuse and fold_se:
                    pw2 = e["pw2"]
                    wimg = torch.empty((N,) + tuple(pw2.tc.shape), dtype=torch.bfloat16, device=dev)
                    self.gate_scale_weights(gap, gap_fixed, d.H * d.W, e["se"], pw2.tc, wimg, pw2.cin, False, e["dw"].name)
                    o = self.new(N, d.H, d.W, pw2.cout)
                    M = N * d.H * d.W
                    res = f if s["identity"] else None
                    self._run("conv_tc", pw2.name, M * (pw2.cin + pw2.cout * (2 if res is not None else 1)) * 2 + wimg.numel() * 2,
                              2 * M * pw2.cout * pw2.cin, self.lib.cabinet_conv_tc_imgw, d.ptr, d.ld, N, d.H, d.W, d.C,
                              wimg.data_ptr(), pw2.tc[0].numel() * pw2.tc.shape[0], pw2.cout, 1, 1, 1, 0, pw2.b.data_ptr(),
                              res.ptr if res is not None else None, res.ld if res is not None else 0, o.ptr, o.dt, o.ld,
                              d.H, d.W, ACT_NONE, self.stream)
                    f = o
                    continue
                scale = self.gate(gap.view(N, -1), d.H * d.W, e["se"], e["dw"].name, gap_fixed)
                # expand form: SE then activation; no-expand form: activation (already applied) then SE (F10)
                se_act = e["act"] if s["expand"] else ACT_NONE
                pw2 = e["pw2"]
                if ((self.fuse_se or e["dw"].name[:-3] in self.fuse_se_blocks) and not self.debug and self.use_tc
                        and pw2.tc is not None and d.dt == BF16 and d.C % 8 == 0):
                    # fused: the project GEMM applies act(x * scale) to its A tiles in shared memory
                    f = self.conv(d, pw2, res=f if s["identity"] else None, a_scale=scale, a_act=se_act)
                    continue
                self.scale_act(d, scale, se_act, e["dw"].name)
            else:
                d, _ = self.dwconv(h, e["dw"])
            f = self.conv(d, e["pw2"], res=f if s["identity"] else None)
        return self.conv(f, self.last, out=out)

    @torch.no_grad()
    def forward_backbone(self, x: torch.Tensor) -> torch.Tensor:
        """Standalone MobileNetV3: (N, 3, H, W) fp32 / bf16 / fp16 -> (N, out_channels, h32, w32) NCHW in x's dtype."""
        N, _, H, W = x.shape
        OH, OW = _out_size(H, 3, 2, 1), _out_size(W, 3, 2, 1)
        h32, w32 = backbone_hw([e["spec"] for e in self.blocks], OH, OW)
        C = self.last.cout
        y = torch.empty((N, C, h32, w32), dtype=x.dtype, device=x.device)
        self.launches = 0
        if N == 0:
            return y
        with self._guard():
            xf = x if x.dtype == torch.float32 and x.is_contiguous() else x.float().contiguous()
            n_se = sum(1 for b in self.blocks if "se" in b)
            gap_all = torch.zeros((max(2 * n_se, 1), N * 1024), dtype=torch.float32, device=self.dev)
            self.launches += 1
            if (self.use_tc and self.use_stem3 and self.stem_tc3 is not None and W % 4 == 0
                    and xf.data_ptr() % 16 == 0):
                f = self.new(N, OH, OW, 16)
                self._run("stem3_tc", "mobile.stem", xf.numel() * 4 + f.t.numel() * 2 + self.stem_tc3.numel() * 2,
                          2 * N * OH * OW * 16 * 27, self.lib.cabinet_stem3_tc, xf.data_ptr(), N, H, W,
                          self.stem_tc3.data_ptr(), f.ptr, f.ld, OH, OW, self.stream)
            else:
                f = self.conv(None, self.stem, nchw_input=xf)
            mf = self.mobilenet(f, gap_all)
            self.relayout(mf.t, (h32 * w32 * C, w32 * C, C, 1), y, (y.stride(0), y.stride(2), y.stride(3), y.stride(1)),
                          N, h32, w32, C, "mobile.out")
        return y

    def spatial_branch(self, s1: Map, out: Optional[Map] = None) -> Map:
        """The SpatialBranch after ``sb.conv1`` (reference: cabinet.py:108-129): sb.conv2, sb.conv3, sb.conv_out.  ``s1``:
        sb.conv1's output; ``out``: where sb.conv_out writes (CABiNet: channels [0:128] of the FFM concat buffer) or None."""
        s2 = self.conv(s1, self.sb2)
        s3 = self.conv(s2, self.sb3)
        return self.conv(s3, self.sb4, out=out)

    def attention_branch(self, cat: Map, n_in: int, low_path=None, need_high: bool = True, high_path=None):
        """AttentionBranch (reference: cabinet.py:75-94).  ``cat``: the b1 concat buffer [x | CAB feat] (cabinet.py:87)
        with x in channels [0:n_in]; the CAB writes the rest.  -> (low, high): ``low_path(feat)`` (default: convb;
        CABiNet's adds its x4 upsample) and b4's fp32 class logits, None unless ``need_high``.  The low path runs on a
        side stream beside b1 -> b4; ``high_path(high)`` is enqueued before the join."""
        feat = self.conv(cat.slice(0, n_in), self.conva)
        feat2 = cat.slice(n_in, feat.C)
        self.cab(feat, feat2)
        if low_path is None:
            low_path = lambda f: self.conv(f, self.convb)  # noqa: E731
        if not need_high:
            return low_path(feat2), None
        with self._branch(0) as joined:  # low-level path beside b1 / b4
            low = low_path(feat2)
            joined(low.t)
        fused = self.conv(cat, self.b1)
        high = self.conv(fused, self.b4, out_dtype=torch.float32)  # class logits stay fp32
        if high_path is not None:
            high_path(high)
        self._join(0)
        return low, high

    def ffm_feat(self, cat: Map, gap: torch.Tensor, scratch: torch.Tensor, low_fold: Optional[Map] = None) -> Map:
        """FeatureFusionModule up to its gate (reference: cabinet.py:142-147): convblk over ``cat`` = [fsp | fcp], and the
        per-(image, channel) sums of its output into ``gap`` [N, C] (``scratch``: zeroed, 128 + N * 64 * C floats).
        ``low_fold``: CABiNet's fp32 1/32-resolution low map, upsampled and added in convblk's epilogue (``fold_low_up``);
        ``cat`` then holds the spatial-branch half only."""
        if low_fold is not None:
            L, (N, H8, W8) = self.ffm_sb, (cat.N, cat.H, cat.W)
            ff = self.new(N, H8, W8, L.cout)
            M = N * H8 * W8
            self._run("conv_tc", L.name, (M * (L.cin + L.cout) + L.w.numel()) * 2 + low_fold.t.numel() * 4,
                      2 * M * L.cout * L.cin, self.lib.cabinet_conv_tc_up, cat.ptr, cat.ld, N, H8, W8, L.cin,
                      L.tc.data_ptr(), L.cout, 1, 1, 1, 0, L.b.data_ptr(), low_fold.ptr, low_fold.H, low_fold.W, ff.ptr,
                      ff.ld, H8, W8, L.act, self.stream)
        else:
            ff = self.conv(cat, self.ffm_blk)
        self.channel_sum(ff, gap, "ffm.gap", scratch)
        return ff

    def ffm_gate_apply(self, ff: Map, gap: torch.Tensor):
        """ff = ff * atten + ff in place, atten = sigmoid(conv2(relu(conv1(mean(ff))))) (reference: cabinet.py:148-153)."""
        att = self.gate(gap, ff.H * ff.W, self.ffm_gate, "ffm.gate")
        self.scale_act(ff, att, ACT_NONE, "ffm.gate", plus_one=True)

    def head(self, f: Map, ffm_gap: Optional[torch.Tensor] = None) -> Map:
        """CABiNetOutput (reference: cabinet.py:162-172) -> its fp32 class map.  ``ffm_gap``: ``f`` is the FFM's convblk
        output with the gate still to apply, and these are its pooling sums (``ffm_feat``)."""
        hcl = self.head_conv
        N, H8, W8 = f.N, f.H, f.W
        if (ffm_gap is not None and self.fold_ffm and self.use_tc and not self.debug and hcl.tc is not None
                and f.dt == BF16 and hcl.kh * hcl.kw > 1):
            # feat * atten + feat is a per-(image, channel) scale of the head conv's INPUT: fold it into per-image
            # copies of the head weights (19 MB) instead of rewriting the 134 MB feature map; the gate MLP runs inside
            # the same launch
            wimg = torch.empty((N,) + tuple(hcl.tc.shape), dtype=torch.bfloat16, device=self.dev)
            self.gate_scale_weights(ffm_gap, False, H8 * W8, self.ffm_gate, hcl.tc, wimg, hcl.cin, True, "ffm.gate")
            hc = self.new(N, H8, W8, hcl.cout)
            M = N * H8 * W8
            self._run("conv_tc", hcl.name, (M * (hcl.cin + hcl.cout) + wimg.numel()) * 2,
                      2 * M * hcl.cout * hcl.cin * hcl.kh * hcl.kw, self.lib.cabinet_conv_tc_imgw, f.ptr, f.ld, N, H8, W8,
                      f.C, wimg.data_ptr(), hcl.tc[0].numel() * hcl.tc.shape[0], hcl.cout, hcl.kh, hcl.kw, hcl.stride,
                      hcl.pad, hcl.b.data_ptr(), None, 0, hc.ptr, hc.dt, hc.ld, H8, W8, hcl.act, self.stream)
        else:
            if ffm_gap is not None:
                self.ffm_gate_apply(f, ffm_gap)
            hc = self.conv(f, hcl)
        return self.conv(hc, self.head_out, out_dtype=torch.float32)

    # ------------------------------------------------------------------ standalone branches and heads
    def _to_map(self, x: torch.Tensor, m: Map, name: str):
        """NCHW ``x`` -> the NHWC map ``m`` (a channel slice of a concat buffer, say), in m's dtype."""
        self.relayout(x, _nchw_strides(x), m.t[..., m.off:m.off + m.C], (m.H * m.W * m.ld, m.W * m.ld, m.ld, 1), m.N, m.H,
                      m.W, m.C, name)

    def _from_map(self, m: Map, dtype: torch.dtype, name: str) -> torch.Tensor:
        """The NHWC map ``m`` -> a new NCHW tensor of ``dtype``."""
        y = torch.empty((m.N, m.C, m.H, m.W), dtype=dtype, device=self.dev)
        self.relayout(m.t[..., m.off:m.off + m.C], (m.H * m.W * m.ld, m.W * m.ld, m.ld, 1), y, _nchw_strides(y), m.N, m.H,
                      m.W, m.C, name)
        return y

    @torch.no_grad()
    def forward_sb(self, x: torch.Tensor) -> torch.Tensor:
        """Standalone SpatialBranch: (N, 3, H, W) fp32 / bf16 / fp16 -> (N, 128, h8, w8) NCHW in x's dtype.  sb.conv1 runs
        on the tensor cores (cabinet_stem7_tc) when W % 4 == 0 in the bf16 precision, else on conv2d_simt."""
        N, _, H, W = x.shape
        OH, OW = _out_size(H, 7, 2, 3), _out_size(W, 7, 2, 3)
        h8, w8 = _out_size(_out_size(OH, 3, 2, 1), 3, 2, 1), _out_size(_out_size(OW, 3, 2, 1), 3, 2, 1)
        self.launches = 0
        if N == 0 or H * W == 0:
            return torch.empty((N, self.sb4.cout, h8, w8), dtype=x.dtype, device=x.device)
        with self._guard():
            xf = x if x.dtype == torch.float32 and x.is_contiguous() else x.float().contiguous()
            if self.use_tc and self.stem_tc7 is not None and W % 4 == 0 and xf.data_ptr() % 16 == 0:
                s1 = self.new(N, OH, OW, 64)
                self._run("stem7_tc", "sb.conv1", xf.numel() * 4 + s1.t.numel() * 2 + self.stem_tc7.numel() * 2,
                          2 * N * OH * OW * 64 * 147, self.lib.cabinet_stem7_tc, xf.data_ptr(), N, H, W,
                          self.stem_tc7.data_ptr(), s1.ptr, s1.ld, OH, OW, self.stream)
            else:
                s1 = self.conv(None, self.sb1, nchw_input=xf)
            return self._from_map(self.spatial_branch(s1), x.dtype, "sb.out")

    @torch.no_grad()
    def forward_ab(self, x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """Standalone AttentionBranch: (N, inplanes, h, w) -> (low, high) = (N, outplanes, h, w), (N, num_classes, h, w)
        NCHW in x's dtype.  x is written straight into the b1 concat buffer; high stays fp32 until the relayout."""
        N, C, h, w = x.shape
        self.launches = 0
        if N == 0 or h * w == 0:
            return tuple(torch.empty((N, L.cout, h, w), dtype=x.dtype, device=x.device) for L in (self.convb, self.b4))
        with self._guard():
            self._scratch = []  # the PSP pools take freshly zeroed scratch
            cat = self.new(N, h, w, C + self.conva.cout)
            self._to_map(x, cat.slice(0, C), "ab.in")
            low, high = self.attention_branch(cat, C)
            return self._from_map(low, x.dtype, "ab.low"), self._from_map(high, x.dtype, "ab.high")

    @torch.no_grad()
    def forward_ffm(self, fsp: torch.Tensor, fcp: torch.Tensor) -> torch.Tensor:
        """Standalone FeatureFusionModule: (N, c1, h, w), (N, c2, h, w) -> (N, out_chan, h, w) = feat * atten + feat, NCHW
        in fsp's dtype.  fsp / fcp are written straight into the two slices of convblk's input."""
        N, c1, h, w = fsp.shape
        c2, C = fcp.shape[1], self.ffm_blk.cout
        self.launches = 0
        if N == 0 or h * w == 0:
            return torch.empty((N, C, h, w), dtype=fsp.dtype, device=fsp.device)
        with self._guard():
            zeros = torch.zeros(N * C + 128 + N * 64 * C, dtype=torch.float32, device=self.dev)  # gap sums + scratch
            self.launches += 1
            cat = self.new(N, h, w, c1 + c2)
            self._to_map(fsp, cat.slice(0, c1), "ffm.in_sp")
            self._to_map(fcp, cat.slice(c1, c2), "ffm.in_cp")
            gap = zeros[: N * C].view(N, C)
            ff = self.ffm_feat(cat, gap, zeros[N * C:])
            self.ffm_gate_apply(ff, gap)
            return self._from_map(ff, fsp.dtype, "ffm.out")

    @torch.no_grad()
    def forward_head(self, x: torch.Tensor) -> torch.Tensor:
        """Standalone CABiNetOutput: (N, in_chan, h, w) -> (N, n_classes, h, w) class logits (not upsampled) in x's dtype;
        fp32 inside until the relayout."""
        N, C, h, w = x.shape
        self.launches = 0
        if N == 0 or h * w == 0:
            return torch.empty((N, self.head_out.cout, h, w), dtype=x.dtype, device=x.device)
        with self._guard():
            f = self.new(N, h, w, C)
            self._to_map(x, f, "conv_out.in")
            return self._from_map(self.head(f), x.dtype, "conv_out.out")

    def bilinear(self, x: Map, out: Map, name: str):
        nbytes = x.N * x.C * (x.H * x.W * x.t.element_size() + out.H * out.W * out.t.element_size())
        self._run("bilinear_nhwc", name, nbytes, 0, self.lib.cabinet_bilinear_nhwc, x.ptr, x.ld, x.dt, out.ptr, out.ld,
                  out.dt, x.N, x.H, x.W, x.C, out.H, out.W, self.stream)

    # ------------------------------------------------------------------ the forward schedule
    def _trunk(self, x: torch.Tensor, need_aux: bool = True):
        """Everything up to the two fp32 class-logit maps: (final8 [N,H/8,W/8,C], aux8 [N,H/8,W/8,C]).

        ``need_aux=False`` (mask / confusion-matrix / probability callers, which only read ``model(x)[0]``,
        evaluate.py:76-78): the auxiliary head ``b1 -> b4 -> x4 upsample`` (cabinet.py:88-93,234-239) is not launched
        and ``aux8`` is None -- it feeds nothing but the second output."""
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()
        if x.device != self.dev:
            raise RuntimeError(f"input on {x.device}, model on {self.dev}")
        N, _, H, W = x.shape
        self.launches = 0
        dev, C = self.dev, self.n_classes
        n_se = sum(1 for b in self.blocks if "se" in b)
        # ONE memset per forward: the SE / FFM pooling sums, and the scratch areas (tickets + parked partial sums) of the
        # deterministic reductions (cabinet_channel_sum, 2 x cabinet_psp_pool)
        kc = self.key_ch
        # (every SE block owns N x 1024 8-byte slots: int64 fixed-point accumulators on the bf16 path, fp32 sums in the
        # parity mode; the FFM pooling row sits behind them)
        n_gap, n_psp, n_ffm = (2 * n_se + 1) * N * 1024, 128 + N * (110 + 256 * kc), 128 + N * 64 * 256
        zeros_all = torch.zeros(n_gap + 2 * n_psp + n_ffm, dtype=torch.float32, device=dev)
        gap_all = zeros_all[:n_gap].view(2 * n_se + 1, N * 1024)
        self._scratch = [zeros_all[n_gap + i * n_psp: n_gap + (i + 1) * n_psp] for i in range(2)]
        ffm_scratch = zeros_all[n_gap + 2 * n_psp:]
        self.launches += 1

        # ---- spatial branch (reference: cabinet.py:108-129) -> channels [0:128] of the FFM concat buffer
        fused_stems = self.use_tc and self.stem_tc is not None and W % 4 == 0
        if fused_stems:
            OH2, OW2 = (H - 1) // 2 + 1, (W - 1) // 2 + 1
            s1, f0 = self.new(N, OH2, OW2, 64), self.new(N, OH2, OW2, 16)
            nbytes = x.numel() * 4 + (s1.t.numel() + f0.t.numel()) * 2 + 80 * 192 * 2
            if self.use_stem2 and self.stem_tc2 is not None:
                self._run("stem_tc", "sb.conv1+mobile.stem", nbytes, 2 * N * OH2 * OW2 * (64 * 147 + 16 * 27),
                          self.lib.cabinet_stem_tc2, x.data_ptr(), N, H, W, self.stem_tc2.data_ptr(), s1.ptr, s1.ld,
                          f0.ptr, f0.ld, OH2, OW2, self.stream)
            else:
                self._run("stem_tc", "sb.conv1+mobile.stem", nbytes, 2 * N * OH2 * OW2 * (64 * 147 + 16 * 27),
                          self.lib.cabinet_stem_tc, x.data_ptr(), N, H, W, self.stem_tc[0].data_ptr(),
                          self.stem_tc[1].data_ptr(), s1.ptr, s1.ld, f0.ptr, f0.ld, OH2, OW2, self.stream)
        else:
            s1 = self.conv(None, self.sb1, nchw_input=x)
        H8, W8 = _out_size(_out_size(s1.H, 3, 2, 1), 3, 2, 1), _out_size(_out_size(s1.W, 3, 2, 1), 3, 2, 1)
        fold_low = (self.fold_low_up and self.use_tc and not self.debug and self.ffm_sb is not None
                    and self.ffm_sb.tc is not None and self.low_fold.tc is not None and self.sb4.cout == self.ffm_sb.cin)
        cat_ffm = self.new(N, H8, W8, self.sb4.cout if fold_low else 128 + 256)
        if self.sb_overlap:  # experiment: the rest of the spatial branch beside the backbone (joined before the FFM)
            with self._branch(2) as joined:
                self.spatial_branch(s1, cat_ffm.slice(0, 128))
                joined(s1.t)
        else:
            self.spatial_branch(s1, cat_ffm.slice(0, 128))

        # ---- backbone (reference: mobilenetv3.py:202-205) -> channels [0:960 | 576] of the b1 concat buffer
        f = f0 if fused_stems else self.conv(None, self.stem, nchw_input=x)
        h32, w32 = backbone_hw([e["spec"] for e in self.blocks], f.H, f.W)
        cat_b1 = self.new(N, h32, w32, self.last.cout + 256)  # [mobile_feat | CAB feat] (reference: cabinet.py:87)
        mf = self.mobilenet(f, gap_all, out=cat_b1.slice(0, self.last.cout))

        # ---- attention branch (reference: cabinet.py:75-94, cab.py:131-162,175-184,213-216)
        def low_path(feat2):
            if fold_low:  # fp32 [N, h32, w32, 256] map that the convblk epilogue upsamples and adds
                return self.conv(feat2, self.low_fold, out_dtype=torch.float32)
            lo = self.conv(feat2, self.convb)
            self.bilinear(lo, cat_ffm.slice(128, 256), "low_up")   # 1/32 -> 1/8 (reference: cabinet.py:228-233)
            return lo

        need_high = need_aux or self.debug
        aux8 = self.new(N, H8, W8, C, torch.float32) if need_high else None
        low, high = self.attention_branch(cat_b1, self.last.cout, low_path, need_high,
                                          lambda hi: self.bilinear(hi, aux8, "high_up"))

        # ---- feature fusion (reference: cabinet.py:142-153)
        self._join(2)
        gap = gap_all[2 * n_se].view(-1)[: N * 256].view(N, 256)
        ff = self.ffm_feat(cat_ffm, gap, ffm_scratch, low if fold_low else None)

        # ---- head (reference: cabinet.py:162-172), the FFM's gate folded into it or applied first
        final8 = self.head(ff, gap)
        if self.debug:  # stage activations for the parity tests (keeps the buffers alive)
            self.stages = dict(feat_sb=cat_ffm.slice(0, 128), mobile_feat=mf, low=low, high=high, feat_fuse=ff,
                               final8=final8, aux8=aux8)
        return final8, aux8

    def _logits(self, x, outs, odt):
        """Trunk + the two x8 upsamples, written into rows of the preallocated NCHW outputs."""
        N, _, H, W = x.shape
        final8, aux8 = self._trunk(x)
        for name, src, y in (("final_up", final8, outs[0]), ("aux_up", aux8, outs[1])):
            nbytes = src.t.numel() * 4 + y.numel() * y.element_size()
            self._run("upsample_logits_nchw", name, nbytes, 0, self.lib.cabinet_upsample_logits_nchw, src.ptr, N,
                      src.H, src.W, src.C, y.data_ptr(), odt, H, W, self.stream)

    def _forward_eager(self, x, out_dtype):
        N, _, H, W = x.shape
        odt = BF16 if out_dtype == torch.bfloat16 else F32
        tdt = torch.bfloat16 if odt == BF16 else torch.float32
        outs = [torch.empty((N, self.n_classes, H, W), dtype=tdt, device=self.dev) for _ in range(2)]
        if N == 0:  # empty batch: nothing to launch
            self.launches = 0
            return outs[0], outs[1]
        if self.dual_stream and N >= 2:
            # two half-batches on two streams (fork / join): the latency-bound low-resolution chain of one half
            # overlaps the bandwidth-bound high-resolution layers of the other
            cur = torch.cuda.current_stream(self.dev)
            if self._side is None:
                self._side = torch.cuda.Stream(self.dev)
            half = N // 2
            self._side.wait_stream(cur)
            self._logits(x[:half], [o[:half] for o in outs], odt)
            launches = self.launches
            with torch.cuda.stream(self._side):
                self._logits(x[half:], [o[half:] for o in outs], odt)
            cur.wait_stream(self._side)
            self.launches += launches
            return outs[0], outs[1]
        chunk = self.sub_batch if self.sub_batch and self.sub_batch < N else N
        launches = 0
        for i in range(0, N, chunk):  # images are independent units: optional L2-sized sub-batches
            self._logits(x[i:i + chunk], [o[i:i + chunk] for o in outs], odt)
            launches += self.launches
        self.launches = launches
        return outs[0], outs[1]

    def _guard(self):
        """The model's GPU as the current device while kernels are enqueued (a model on a non-current GPU would
        otherwise launch in the wrong device context)."""
        import contextlib

        return torch.cuda.device(self.dev) if torch.device(self.dev).type == "cuda" else contextlib.nullcontext()

    @torch.no_grad()
    def forward(self, x, out_dtype=torch.float32):
        with self._guard():
            return self._forward(x, out_dtype)

    def _forward(self, x, out_dtype=torch.float32):
        """-> (final_logit, high_res_logit_up) NCHW (reference: cabinet.py:240-247).

        With ``use_cuda_graph`` the whole kernel schedule of a given input shape is captured once and replayed; the
        returned tensors are then the graph's static output buffers (overwritten by the next call of that shape)."""
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()
        if not self.use_cuda_graph or self.trace is not None or self.debug or x.shape[0] == 0:
            return self._forward_eager(x, out_dtype)
        key = (tuple(x.shape), out_dtype, self.sub_batch, self.dual_stream)
        # A caller that keeps feeding the SAME buffer (an evaluator's device-side input slot, a benchmark) gets a graph
        # captured on that address: no 2 x 201 MB staging copy per call.  Anything else goes through a static input
        # buffer.  All graphs of the engine share one memory pool.
        pkey = key + (x.data_ptr(),)
        g = self._graphs.get(pkey)
        if g is None:
            if len(self._graph_seen) > 4096:
                self._graph_seen.clear()
            seen = self._graph_seen.get(pkey, 0) + 1
            self._graph_seen[pkey] = seen
            if seen >= 3 and sum(1 for k in self._graphs if len(k) == len(pkey)) < 4:
                g = self._capture_forward(x, out_dtype)
                self._graphs[pkey] = g
            else:
                g = self._graphs.get(key)
                if g is None:
                    g = self._capture_forward(x.clone(), out_dtype)
                    self._graphs[key] = g
        graph, static_x, outs, launches = g
        if x.data_ptr() != static_x.data_ptr():
            static_x.copy_(x, non_blocking=True)
        graph.replay()
        self.launches = launches
        return outs

    def _capture_forward(self, static_x, out_dtype):
        cur = torch.cuda.current_stream(self.dev)
        side = torch.cuda.Stream(self.dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):  # warm-up outside capture (lazy function attributes, allocator)
            self._forward_eager(static_x, out_dtype)
        cur.wait_stream(side)
        if self._pool is None:
            self._pool = torch.cuda.graph_pool_handle()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, pool=self._pool):
            outs = self._forward_eager(static_x, out_dtype)
        return (graph, static_x, outs, self.launches)

    def _argmax(self, final8: Map, N, H, W, labels=None, hist=None, ignore_label=255):
        mask = torch.empty((N, H, W), dtype=torch.uint8, device=self.dev)
        nbytes = final8.t.numel() * 4 + mask.numel() + (labels.numel() * labels.element_size() if labels is not None else 0)
        self._run("upsample_argmax", "mask" if hist is None else "mask+hist", nbytes, 0,
                  self.lib.cabinet_upsample_argmax, final8.ptr, N, final8.H, final8.W, final8.C, mask.data_ptr(), H, W,
                  labels.data_ptr() if labels is not None else None,
                  0 if labels is None or labels.dtype == torch.int64 else 1, ignore_label,
                  hist.data_ptr() if hist is not None else None, self.stream)
        return mask

    def _graphed(self, key, fn):
        """Run ``fn`` eagerly the first time a key (shapes + buffer addresses) is seen, capture it into a CUDA graph
        the second time, replay afterwards.  ``fn`` must only touch the buffers named in the key."""
        if not self.use_cuda_graph or self.trace is not None or self.debug:
            return fn()
        g = self._graphs.get(key)
        if g is None:
            if len(self._graph_seen) > 4096:  # callers that never repeat a buffer: do not grow without bound
                self._graph_seen.clear()
            seen = self._graph_seen.get(key, 0) + 1
            self._graph_seen[key] = seen
            if seen < 2 or len(self._graphs) >= 16:
                return fn()
            if self._pool is None:
                self._pool = torch.cuda.graph_pool_handle()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, pool=self._pool):  # one activation pool for all graphs of this engine
                out = fn()
            g = (graph, out, self.launches)
            self._graphs[key] = g
        graph, out, launches = g
        graph.replay()
        self.launches = launches
        return out

    @torch.no_grad()
    def forward_mask(self, x):
        N, _, H, W = x.shape
        if N == 0:
            return torch.empty((0, H, W), dtype=torch.uint8, device=self.dev)
        with self._guard():
            final8, _ = self._trunk(x, need_aux=False)
            return self._argmax(final8, N, H, W)

    @torch.no_grad()
    def class_map8(self, x):
        """(N,3,H,W) -> fp32 NHWC class map (N, H/8, W/8, C): ``conv_out(feat_fuse)`` before the final x8 bilinear
        (reference: cabinet.py:236-243).  What the evaluator's fused softmax / accumulate tail consumes; the auxiliary
        head is not computed.  A repeated input buffer (the evaluator's chip slots) is captured into a CUDA graph; the
        returned tensor is then that graph's output buffer (overwritten by the next call with the same input buffer)."""
        N, _, H, W = x.shape
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()

        def run():
            return self._trunk(x, need_aux=False)[0].t

        with self._guard():
            return self._graphed(("cls8", tuple(x.shape), x.data_ptr()), run)

    @torch.no_grad()
    def forward_hist(self, x, labels, hist, ignore_label=255):
        N, _, H, W = x.shape
        if labels.dim() == 4:
            labels = labels.squeeze(1)
        if labels.dtype not in (torch.int64, torch.uint8) or labels.device != self.dev or not labels.is_contiguous():
            raise ValueError("labels must be a contiguous int64/uint8 (N,H,W) tensor on the model's device")
        if hist.dtype != torch.int64 or tuple(hist.shape) != (self.n_classes, self.n_classes) or hist.device != self.dev:
            raise ValueError("hist must be an int64 (C,C) tensor on the model's device")
        if tuple(labels.shape) != (N, H, W):
            raise ValueError(f"labels shape {tuple(labels.shape)} != {(N, H, W)}")
        if N == 0:
            return torch.empty((0, H, W), dtype=torch.uint8, device=self.dev)
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()

        def run():
            final8, _ = self._trunk(x, need_aux=False)
            return self._argmax(final8, N, H, W, labels, hist, ignore_label)

        # static buffers (an evaluator's double-buffered device tensors) -> captured once, replayed afterwards
        with self._guard():
            return self._graphed(("hist", tuple(x.shape), x.data_ptr(), labels.data_ptr(), labels.dtype, hist.data_ptr(),
                                  ignore_label), run)

    # ------------------------------------------------------------------ tracing (bench / profiles)
    def start_trace(self, kernels=None):
        """Bracket every launch (or only the named kernels) with CUDA events until ``stop_trace``."""
        self.trace, self.trace_filter = [], (set(kernels) if kernels else None)

    def stop_trace(self):
        """-> list of dict(kernel, layer, bytes, flops, ms); synchronises."""
        torch.cuda.synchronize(self.dev)
        rows = [dict(kernel=k, layer=l, bytes=b, flops=f, ms=e0.elapsed_time(e1), fused_bytes=fb)
                for k, l, b, f, e0, e1, fb in self.trace]
        self.trace = None
        return rows

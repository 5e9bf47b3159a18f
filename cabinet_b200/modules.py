"""Parameter tree of the CABiNet drop-in.

The classes here are *containers*: they own exactly the parameters/buffers the
reference model owns, under exactly the reference's names, created and
initialised in exactly the reference's order (so the same ``torch.manual_seed``
gives bit-identical weights), but they hold no arithmetic.  All arithmetic of
``CABiNet.forward`` lives in the sm_100a kernels reached through
``cabinet_b200.engine`` -> ``libcabinet_b200.so`` (C-ABI).

Reference surface mirrored (names/shapes/order only):
  src/models/mobilenetv3.py:68-83,86-99,102-159,162-235   (SE, stems, MBConv, backbone + init)
  src/models/cab.py:18-38,46-76,84-129,170-184,192-211    (DWConv, PSP, global/local attention, CAB)
  src/models/cabinet.py:19-51,54-105,108-129,132-140,156-160,175-205,249-300
"""

from __future__ import annotations

import copy
import math
from pathlib import Path
from typing import Optional, Tuple

import torch
from torch import nn

from .constants import BACKBONE_CFGS, MODEL_CONFIG, PSP_SIZES, make_divisible, resolve_blocks


def _slot() -> nn.Module:
    """Index filler for a parameter-free position of a reference ``nn.Sequential``."""
    return nn.Identity()


def _conv(cin, cout, k=1, s=1, p=0, groups=1, bias=False) -> nn.Conv2d:
    return nn.Conv2d(cin, cout, k, s, p, groups=groups, bias=bias)


# --------------------------------------------------------------------------- backbone
class SqueezeExcite(nn.Module):
    """Holds ``fc.0`` / ``fc.2`` (reference: mobilenetv3.py:68-77)."""

    def __init__(self, channels: int):
        super().__init__()
        hidden = make_divisible(channels // 4, 8)
        self.fc = nn.Sequential(nn.Linear(channels, hidden), _slot(), nn.Linear(hidden, channels), _slot())


class MBConv(nn.Module):
    """Holds the ``conv.N`` slots of one inverted-residual block (reference: mobilenetv3.py:102-153).

    Slot layout (F10): expand form ``0 pw,1 bn,3 dw,4 bn,5 se,7 pw,8 bn``;
    no-expand form ``0 dw,1 bn,3 se,4 pw,5 bn``.
    """

    def __init__(self, inp, hidden, oup, k, stride, use_se, use_hs):
        super().__init__()
        if stride not in (1, 2):
            raise ValueError(f"stride must be 1 or 2, got {stride}")
        self.spec = dict(inp=inp, exp=hidden, out=oup, k=k, s=stride, se=bool(use_se), hs=bool(use_hs),
                         identity=(stride == 1 and inp == oup), expand=(inp != hidden))
        dw = lambda: _conv(hidden, hidden, k, stride, (k - 1) // 2, groups=hidden)  # noqa: E731
        se = lambda: SqueezeExcite(hidden) if use_se else _slot()  # noqa: E731
        if inp == hidden:
            seq = [dw(), nn.BatchNorm2d(hidden), _slot(), se(), _conv(hidden, oup), nn.BatchNorm2d(oup)]
        else:
            seq = [_conv(inp, hidden), nn.BatchNorm2d(hidden), _slot(), dw(), nn.BatchNorm2d(hidden), se(), _slot(),
                   _conv(hidden, oup), nn.BatchNorm2d(oup)]
        self.conv = nn.Sequential(*seq)


class MobileNetV3(nn.Module):
    """Backbone parameter tree (reference: mobilenetv3.py:162-235)."""

    def __init__(self, cfgs, mode, num_classes=1000, width_mult=1.0, weights=None):
        super().__init__()
        self.cfgs = cfgs
        self.weights = weights
        if mode not in ("large", "small"):
            raise ValueError(f"mode must be 'large' or 'small', got '{mode}'")
        stem, blocks, last_exp = resolve_blocks(cfgs, width_mult)
        feats = [nn.Sequential(_conv(3, stem, 3, 2, 1), nn.BatchNorm2d(stem), _slot())]
        for b in blocks:
            feats.append(MBConv(b["inp"], b["exp"], b["out"], b["k"], b["s"], b["se"], b["hs"]))
        self.features = nn.Sequential(*feats)
        last_in = blocks[-1]["out"] if blocks else stem
        self.conv = nn.Sequential(_conv(last_in, last_exp), nn.BatchNorm2d(last_exp), _slot())
        self.avgpool = _slot()  # parameter-free in the reference as well; unused by forward (F9)
        head = MODEL_CONFIG[mode]["output_channel"]
        if width_mult > 1.0:
            head = make_divisible(head * width_mult, 8)
        # classifier.{0,3}: in the state_dict, never used by the forward path (F9)
        self.classifier = nn.Sequential(nn.Linear(last_exp, head), _slot(), _slot(), nn.Linear(head, num_classes))
        self.out_channels = last_exp
        self._initialize_weights()

    def _initialize_weights(self):
        """Pretrained load (minus classifier) or the MobileNetV3 init (reference: mobilenetv3.py:207-235)."""
        if self.weights is not None and Path(self.weights).is_file():
            try:
                blob = torch.load(self.weights, map_location="cpu", weights_only=True)
                merged = self.state_dict()
                merged.update({k: v for k, v in blob.items() if "classifier" not in k})
                self.load_state_dict(merged)
                print(f"Loaded pretrained weights from {self.weights}")
                return
            except Exception as e:  # non-fatal in the reference too (mobilenetv3.py:221-223)
                print(f"Failed to load backbone weights from {self.weights}: {e}")
                print("Proceeding with random weight initialization.")
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                fan = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2.0 / fan))
                if m.bias is not None:
                    m.bias.data.zero_()
            elif isinstance(m, nn.BatchNorm2d):
                m.weight.data.fill_(1)
                m.bias.data.zero_()
            elif isinstance(m, nn.Linear):
                m.weight.data.normal_(0, 0.01)
                m.bias.data.zero_()


# --------------------------------------------------------------------------- CAB
class DWConv(nn.Module):
    """``block.{0,1}``: depthwise 3x3 + BN (+ReLU) (reference: cab.py:18-38)."""

    def __init__(self, channels, stride=1):
        super().__init__()
        self.block = nn.Sequential(_conv(channels, channels, 3, stride, 1, groups=channels),
                                   nn.BatchNorm2d(channels), _slot())


class PSPModule(nn.Module):
    """``project``: bias-free 1x1 over [x, up(pool_s(x))...] (reference: cab.py:46-63)."""

    def __init__(self, in_channels, sizes=PSP_SIZES):
        super().__init__()
        self.sizes = tuple(sizes)
        self.stages = nn.ModuleList([_slot() for _ in sizes])
        self.project = _conv(in_channels * (len(sizes) + 1), in_channels)


class GlobalContextAttention(nn.Module):
    """q/k/v projections + PSP encoders + output projection (reference: cab.py:84-129)."""

    def __init__(self, in_channels, key_channels, value_channels, out_channels=None, scale=1, psp_sizes=PSP_SIZES):
        super().__init__()
        if scale != 1:
            raise ValueError("only scale=1 is on the CABiNet forward path (reference: cab.py:203-209)")
        self.scale = scale
        self.out_channels = out_channels or in_channels
        self.pool = _slot()
        self.to_query = nn.Sequential(_conv(in_channels, key_channels), nn.BatchNorm2d(key_channels), _slot())
        self.to_key = nn.Sequential(_conv(in_channels, key_channels), nn.BatchNorm2d(key_channels), _slot())
        self.to_value = _conv(in_channels, value_channels)
        self.psp_key = PSPModule(key_channels, psp_sizes)
        self.psp_value = PSPModule(value_channels, psp_sizes)
        self.project_out = _conv(value_channels, self.out_channels)
        nn.init.constant_(self.project_out.weight, 0)  # overwritten by AttentionBranch.init_weight (F6)


class LocalAttention(nn.Module):
    def __init__(self, channels):
        super().__init__()
        self.refine = nn.Sequential(DWConv(channels), DWConv(channels), DWConv(channels))
        self.gate = _slot()


class ContextAggregationBlock(nn.Module):
    """gamma * global + local (reference: cab.py:192-211)."""

    def __init__(self, in_channels, value_channels):
        super().__init__()
        self.global_attn = GlobalContextAttention(in_channels, in_channels // 2, value_channels, in_channels, 1)
        self.local_attn = LocalAttention(in_channels)
        self.gamma = nn.Parameter(torch.zeros(1))


# --------------------------------------------------------------------------- CABiNet heads
class ConvBNReLU(nn.Module):
    """``conv`` + ``bn`` (reference: cabinet.py:19-51)."""

    def __init__(self, in_chan, out_chan, kernel_size=3, stride=1, padding=1, dilation=1):
        super().__init__()
        self.conv = nn.Conv2d(in_chan, out_chan, kernel_size, stride, padding, dilation=dilation, bias=False)
        self.bn = nn.BatchNorm2d(out_chan)
        self.relu = _slot()
        nn.init.kaiming_normal_(self.conv.weight, a=1)


class AttentionBranch(nn.Module):
    """reference: cabinet.py:54-105."""

    def __init__(self, inplanes, interplanes, outplanes, num_classes):
        super().__init__()
        self.conva = nn.Sequential(_conv(inplanes, interplanes, 3, 1, 1), nn.BatchNorm2d(interplanes), _slot())
        self.a2block = ContextAggregationBlock(interplanes, interplanes // 2)
        self.convb = _conv(interplanes, outplanes, bias=True)
        self.b1 = _conv(inplanes + outplanes, outplanes, 3, 1, 1)
        self.b2 = nn.BatchNorm2d(outplanes)
        self.b3 = _slot()
        self.b4 = _conv(outplanes, num_classes, bias=True)
        for m in self.modules():  # re-initialises project_out too (F6)
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, a=1)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)


class SpatialBranch(nn.Module):
    """reference: cabinet.py:108-114."""

    def __init__(self):
        super().__init__()
        self.conv1 = ConvBNReLU(3, 64, 7, 2, 3)
        self.conv2 = ConvBNReLU(64, 64, 3, 2, 1)
        self.conv3 = ConvBNReLU(64, 64, 3, 2, 1)
        self.conv_out = ConvBNReLU(64, 128, 1, 1, 0)


class FeatureFusionModule(nn.Module):
    """reference: cabinet.py:132-140."""

    def __init__(self, in_chan, out_chan):
        super().__init__()
        self.convblk = ConvBNReLU(in_chan, out_chan, 1, 1, 0)
        self.avg_pool = _slot()
        self.conv1 = _conv(out_chan, out_chan // 4)
        self.relu = _slot()
        self.conv2 = _conv(out_chan // 4, out_chan)
        self.sigmoid = _slot()


class CABiNetOutput(nn.Module):
    """reference: cabinet.py:156-160."""

    def __init__(self, in_chan, mid_chan, n_classes):
        super().__init__()
        self.conv = ConvBNReLU(in_chan, mid_chan, 3, 1, 1)
        self.conv_out = _conv(mid_chan, n_classes)


class CABiNet(nn.Module):
    """Drop-in for the reference ``CABiNet`` (reference: cabinet.py:175-300).

    Same constructor, same children (``mobile / ab / sb / ffm / conv_out``), same
    ``state_dict`` keys, ``attention_planes`` and ``get_params()``.  ``forward`` runs the
    sm_100a engine; there is no ATen/CPU fallback: a CPU tensor, a CPU model or a
    missing ``libcabinet_b200.so`` raises.

    Extra (non-reference) knobs, all attributes so the constructor stays identical:
      ``precision``     "bf16" (tcgen05 path, default) or "fp32" (CUDA-core parity mode)
      ``logits_dtype``  dtype of the two returned NCHW logit tensors (default fp32 like the reference)
      ``use_cuda_graph`` / ``sub_batch``  replay a captured schedule / process the batch in L2-sized chunks
    """

    def __init__(self, n_classes: int, backbone_weights: Optional[Path] = None, cfgs=None, mode="large"):
        super().__init__()
        if cfgs is None and mode in BACKBONE_CFGS:
            cfgs = BACKBONE_CFGS[mode]
        cfgs = [list(r) for r in cfgs] if cfgs is not None else cfgs  # list-of-lists or OmegaConf ListConfig
        self.mobile = MobileNetV3(cfgs=cfgs, mode=mode, num_classes=n_classes, weights=backbone_weights)
        config = MODEL_CONFIG.get(mode)
        if config is None:
            raise ValueError(f"Invalid mode: {mode}. Must be 'large' or 'small'")
        self.attention_planes = config["attention_planes"]
        self.n_classes = n_classes
        self.mode = mode
        self.ab = AttentionBranch(self.attention_planes, 256, 256, n_classes)
        self.sb = SpatialBranch()
        self.ffm = FeatureFusionModule(128 + 256, 256)
        self.conv_out = CABiNetOutput(256, 256, n_classes)
        self.precision = "bf16"
        self.logits_dtype = torch.float32
        self.train_precision = "fp32"   # activation dtype of the training step: "fp32" | "bf16" | "fp16"
        self.use_cuda_graph = False  # replay a captured kernel schedule per input shape (static output buffers)
        self.sub_batch = 0           # > 0: run the schedule over chunks of this many images (L2-resident activations)
        self.__dict__["_engine"] = None
        self.__dict__["_train_engine"] = None

    # ------------------------------------------------------------------ engine plumbing
    def _weights_stamp(self):
        return tuple((t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers()))

    def engine(self):
        """The packed-weight execution engine for the current weights/device/precision (lazy, cached)."""
        from .engine import Engine

        eng = self.__dict__.get("_engine")
        stamp = (self.precision, self._weights_stamp())
        if eng is None or eng.stamp != stamp:
            eng = Engine(self, precision=self.precision)
            eng.stamp = stamp
            self.__dict__["_engine"] = eng
        eng.use_cuda_graph, eng.sub_batch = bool(self.use_cuda_graph), int(self.sub_batch)
        return eng

    def repack(self):
        """Drop packed weights (call after mutating parameters through ``.data`` views the stamp cannot see)."""
        self.__dict__["_engine"] = None

    def _apply(self, fn, *a, **kw):
        self.__dict__["_engine"] = None
        self.__dict__["_train_engine"] = None
        return super()._apply(fn, *a, **kw)

    def __deepcopy__(self, memo):  # EMA deep-copies the model (reference: src/utils/ema.py:44)
        eng, teng = self.__dict__.pop("_engine", None), self.__dict__.pop("_train_engine", None)
        try:
            cls = self.__class__
            new = cls.__new__(cls)
            memo[id(self)] = new
            new.__dict__.update({k: copy.deepcopy(v, memo) for k, v in self.__dict__.items()})
            new.__dict__["_engine"] = new.__dict__["_train_engine"] = None
        finally:
            self.__dict__["_engine"], self.__dict__["_train_engine"] = eng, teng
        return new

    def __getstate__(self):
        d = dict(self.__dict__)
        d["_engine"] = d["_train_engine"] = None
        return d

    # ------------------------------------------------------------------ forward surface
    def _check_input(self, x, inference_only=True):
        if not isinstance(x, torch.Tensor) or x.dim() != 4 or x.shape[1] != 3:
            raise ValueError(f"expected an (N, 3, H, W) tensor, got {getattr(x, 'shape', type(x))}")
        if not x.is_cuda:
            raise RuntimeError("cabinet_b200.CABiNet has no CPU path: move the model and the input to a CUDA device")
        if self.training and inference_only:
            raise RuntimeError("the fused mask / confusion-matrix / class-map calls are inference paths (eval-mode BN); "
                               "call .eval() first")

    def train_engine(self):
        """The training-step engine (train-mode forward + backward kernels) for the current device / precision."""
        from .train_engine import TrainEngine

        eng = self.__dict__.get("_train_engine")
        dev = next(self.parameters()).device
        if eng is None or eng.dev != dev or eng.precision != self.train_precision:
            eng = self.__dict__["_train_engine"] = TrainEngine(self, precision=self.train_precision)
        return eng

    def forward(self, x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """(N,3,H,W) -> (final_logit, high_res_logit_up), each (N, n_classes, H, W) NCHW.

        reference: cabinet.py:207-247 (the aux head is upsampled in two stages, F8).  ``.eval()``: the inference
        schedule (BN folded into the weights).  ``.train()``: batch-statistics BatchNorm (running statistics updated) and a
        differentiable result -- ``loss.backward()`` fills ``p.grad`` of every parameter on the forward path
        (reference: src/scripts/train.py:429-441); ``torch.no_grad()`` in train mode gives the same forward without a tape
        kept alive (``val_step``, train.py:443-456).  Partial fine-tuning works as with an ``nn.Module``: a parameter with
        ``requires_grad=False`` gets no gradient (and layers that lead to no trainable parameter run no backward), and
        a BatchNorm put in ``.eval()`` uses and keeps its running statistics.

        Input gradients: an ``x`` that requires grad gets ``x.grad`` in both modes.  In ``.eval()`` with grad mode on and
        ``x.requires_grad`` (adversarial attacks, saliency, a frozen segmenter as a loss), the call runs the
        differentiable training schedule at ``train_precision`` with every BatchNorm in eval mode: running-statistics
        normalisation, buffers untouched, gradients for the parameters that require grad and for ``x``.  Every other
        eval-mode call (``x`` without grad, ``torch.no_grad()``, ``torch.inference_mode()``) stays on the inference
        schedule and returns outputs without ``grad_fn``.
        """
        if self.training or (torch.is_grad_enabled() and x.requires_grad):
            self._check_input(x, inference_only=False)
            from .train_engine import TrainStep

            params = [p for n, p in self.named_parameters() if not n.startswith("mobile.classifier")]
            return TrainStep.apply(self.train_engine(), self.logits_dtype, x, *params)
        self._check_input(x)
        return self.engine().forward(x, out_dtype=self.logits_dtype)

    @torch.no_grad()
    def predict_mask(self, x: torch.Tensor) -> torch.Tensor:
        """(N,3,H,W) -> uint8 (N,H,W) argmax of ``final_logit`` (fused upsample+argmax, logits never hit HBM).

        Equals ``torch.argmax(model(x)[0], dim=1)`` of the fast eval mode (reference: evaluate.py:76-78,222).
        """
        self._check_input(x)
        return self.engine().forward_mask(x)

    @torch.no_grad()
    def accumulate_hist(self, x: torch.Tensor, labels: torch.Tensor, hist: torch.Tensor, ignore_label: int = 255):
        """Fused forward -> argmax -> ``hist[pred, label] += 1`` into an int64 (C,C) device tensor.

        reference: evaluate.py:162-191,222-228 (orientation hist[pred, label], ignore, clip).
        """
        self._check_input(x)
        return self.engine().forward_hist(x, labels, hist, ignore_label)

    @torch.no_grad()
    def class_map8(self, x: torch.Tensor) -> torch.Tensor:
        """(N,3,H,W) -> fp32 NHWC (N, H/8, W/8, n_classes) class map of the head, i.e. ``final_logit`` before its
        x8 bilinear upsample (reference: cabinet.py:236-243).  Input of ``cabinet_upsample_softmax_accum``."""
        self._check_input(x)
        if x.shape[0] == 0:
            raise ValueError("class_map8 needs a non-empty batch")
        return self.engine().class_map8(x)

    # ------------------------------------------------------------------ optimizer surface
    def get_params(self):
        """(wd, nowd, lr_mul_wd, lr_mul_nowd) with ``ab / ffm / conv_out`` as the x10-LR decoder.

        reference: cabinet.py:249-300 (consumed by src/utils/optimizer.py:56-101).
        """
        groups = {False: ([], []), True: ([], [])}
        for name, child in self.named_children():
            wd, nowd = groups[name in ("ffm", "conv_out", "ab")]
            seen = set()
            for m in child.modules():
                if isinstance(m, nn.Conv2d):
                    wd.append(m.weight)
                    seen.add(id(m.weight))
                    if m.bias is not None:
                        nowd.append(m.bias)
                        seen.add(id(m.bias))
                elif isinstance(m, nn.BatchNorm2d):
                    for p in m.parameters():
                        nowd.append(p)
                        seen.add(id(p))
            nowd.extend(p for p in child.parameters() if id(p) not in seen)  # Linear (SE), gamma
        return groups[False][0], groups[False][1], groups[True][0], groups[True][1]

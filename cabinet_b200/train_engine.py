"""Training step of the drop-in model (BASELINE config 5): train-mode forward + backward on the C-ABI kernels.

reference: ``src/scripts/train.py:429-441`` -- ``out, out16 = net(im)`` with the model in ``.train()`` (batch-statistics
BatchNorm, running statistics updated), two ``OhemCELoss`` terms, ``loss.backward()``.  ``cabinet_b200.CABiNet`` in
train mode routes ``forward`` through :class:`TrainStep` (a ``torch.autograd.Function``): its forward runs the schedule
below and keeps a tape of the tensors the backward kernels need; its backward receives the gradients of the two logit
tensors and returns one fp32 gradient per parameter, so ``loss.backward()``, ``GradScaler`` and optimizers work as with
the reference module.  PyTorch supplies memory, streams and the autograd hand-off only: every arithmetic step is a
kernel of ``libcabinet_b200.so`` (``csrc/train.cu`` + the forward kernels of the inference path).

Layout: NHWC activations (fp32 in ``precision='fp32'``, bf16 in ``'bf16'``, fp16 in ``'fp16'``), class-logit maps /
statistics / parameter gradients fp32.  ``'fp16'`` is the ``'bf16'`` schedule with fp16 storage and fp16 tensor-core
operands: the numerics of the reference's ``autocast`` + ``GradScaler`` recipe (an overflow reaches the parameter
gradients as inf / NaN, so ``GradScaler`` skips the step).  All reductions are deterministic (fixed summation order), so a step is bit-reproducible.

Partial fine-tuning follows PyTorch per module: a parameter with ``requires_grad=False`` gets no gradient, a layer whose
input and parameters need none runs no backward, and a BatchNorm in eval mode uses (and keeps) its running statistics.
An input that requires grad gets its gradient: both stems' output gradients are then computed (even for frozen stem
weights) and one ``cabinet_stem_dgrad`` call turns them into the fp32 NCHW ``dx``.

The step is ~660 C-ABI calls; enqueueing them from Python takes ~19 ms against ~21 ms of GPU work, and the small layers
at the end of the network leave the GPU waiting for the host.  After ``graph_after`` eager steps with the same input
geometry the engine therefore captures the forward and the backward schedule into two CUDA graphs that share one
memory pool (static input / logit / logit-gradient / parameter-gradient buffers) and replays them: same kernels, same
order, same results, two graph launches per step.  A changed parameter or buffer address (``.to()``, ``.half()``), input
shape or engine switch re-captures; tracing (``start_trace``) and steps inside someone else's capture stay eager.
"""

from __future__ import annotations

import contextlib
import gc
import math
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import ACT_HSIGMOID, ACT_HSWISH, ACT_NONE, ACT_RELU, ACT_SIGMOID, BF16, F16, F32, check
from .constants import BN_EPS
from .engine import Map, _out_size, backbone_hw, dtype_code

def _sb_hw(H: int, W: int) -> Tuple[int, int]:
    """(h, w) of the spatial branch's output: three stride-2 convolutions (7x7 pad 3, then 3x3 pad 1 twice)."""
    return tuple(_out_size(_out_size(_out_size(n, 7, 2, 3), 3, 2, 1), 3, 2, 1) for n in (H, W))


BN_MOMENTUM = 0.1  # nn.BatchNorm2d default (the reference never overrides it)
PSP_SIZES = (1, 3, 6, 8)  # reference: src/models/cab.py:49


# ----------------------------------------------------------------------------- separable resampling operators (host)
def bilinear_matrix(n_in: int, n_out: int) -> np.ndarray:
    """[n_out][n_in] row operator of F.interpolate(mode='bilinear', align_corners=False) along one axis
    (ATen area_pixel_compute_source_index; reference call sites cabinet.py:228-245, cab.py:70-72)."""
    m = np.zeros((n_out, n_in), dtype=np.float64)
    scale = np.float32(n_in) / np.float32(n_out)
    for o in range(n_out):
        src = max(np.float32((np.float32(o) + np.float32(0.5)) * scale - np.float32(0.5)), np.float32(0.0))
        i0 = min(int(src), n_in - 1)
        i1 = min(i0 + 1, n_in - 1)
        w1 = np.float32(src - np.float32(i0))
        m[o, i0] += float(np.float32(1.0) - w1)
        m[o, i1] += float(w1)
    return m


def adaptive_pool_matrix(n_in: int, n_out: int) -> np.ndarray:
    """[n_out][n_in] row operator of nn.AdaptiveAvgPool2d along one axis (bins floor(b*in/out) .. ceil((b+1)*in/out))."""
    m = np.zeros((n_out, n_in), dtype=np.float64)
    for b in range(n_out):
        lo, hi = (b * n_in) // n_out, -((-(b + 1) * n_in) // n_out)
        m[b, lo:hi] = 1.0 / (hi - lo)
    return m


def csr(mat: np.ndarray):
    """dense [O][I] -> (start int32 [O+1], index int32 [nnz], weight fp32 [nnz])."""
    start, idx, w = [0], [], []
    for row in mat:
        nz = np.nonzero(row)[0]
        idx.extend(nz.tolist())
        w.extend(row[nz].tolist())
        start.append(len(idx))
    return (np.asarray(start, np.int32), np.asarray(idx if idx else [0], np.int32), np.asarray(w if w else [0.0], np.float32))


class _Tables:
    def __init__(self, dev):
        self.dev, self.cache = dev, {}

    def get(self, kind: str, n_in: int, n_out: int, transpose: bool):
        key = (kind, n_in, n_out, transpose)
        if key not in self.cache:
            if kind == "identity":
                m = np.eye(n_in, dtype=np.float64)
            else:
                m = bilinear_matrix(n_in, n_out) if kind == "bilinear" else adaptive_pool_matrix(n_in, n_out)
            s, i, w = csr(m.T if transpose else m)
            self.cache[key] = tuple(torch.from_numpy(a).to(self.dev) for a in (s, i, w))
        return self.cache[key]


class _Grads:
    """Gradient buffers mirror the geometry of the activation buffers (same base tensor shape, so channel slices of a
    concat buffer address the same way); a region written for the first time is overwritten, later writers accumulate."""

    def __init__(self, eng):
        self.eng, self.buf, self.written = eng, {}, {}

    def _base(self, m: Map) -> torch.Tensor:
        k = id(m.t)
        if k not in self.buf:
            self.buf[k] = torch.empty_like(m.t)
            self.written[k] = []
        return self.buf[k]

    def out(self, m: Map) -> Tuple[Map, int]:
        """-> (gradient view of ``m``, accumulate flag) and marks the region written."""
        b = self._base(m)
        spans = self.written[id(m.t)]
        lo, hi = m.off, m.off + m.C
        covered = any(a <= lo and hi <= z for a, z in spans)
        if not covered:
            assert not any(a < hi and lo < z for a, z in spans), "partially overlapping gradient regions"
            spans.append((lo, hi))
        return Map(b, m.N, m.H, m.W, m.C, m.ld, m.off), int(covered)

    def get(self, m: Map) -> Optional[Map]:
        """gradient view of ``m`` if any consumer wrote it."""
        k = id(m.t)
        if k not in self.buf or not any(a <= m.off and m.off + m.C <= z for a, z in self.written[k]):
            return None
        return Map(self.buf[k], m.N, m.H, m.W, m.C, m.ld, m.off)


class TrainEngine:
    def __init__(self, model, precision: str = "fp32"):
        if precision not in ("bf16", "fp16", "fp32"):
            raise ValueError(f"precision must be 'bf16', 'fp16' or 'fp32', got {precision!r}")
        p0 = next(model.parameters())
        if not p0.is_cuda:
            raise RuntimeError("cabinet_b200 training needs the model on a CUDA device (no CPU path)")
        self.lib = _lib.load()
        self.model, self.dev, self.precision = model, p0.device, precision
        # the activation dtype, in one place: every 2-byte buffer and operand of the schedule follows it
        self.tdt = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[precision]
        self.dt = dtype_code(self.tdt)
        # 0: a standalone ContextAggregationBlock (``block_forward``) or MobileNetV3 (``backbone_forward``)
        self.n_classes = getattr(model, "n_classes", 0)
        self.tables = _Tables(self.dev)
        self.tape: List = []
        self.pgrads: Dict[int, torch.Tensor] = {}
        self._pflat: Optional[torch.Tensor] = None   # flat fp32 storage of this backward's parameter gradients
        self._pslots: Dict[int, Tuple[int, int]] = {}
        self._bn_seen: List[torch.Tensor] = []
        self.launches = 0
        self.trace, self.phase = None, "fwd"
        self.use_tc = precision != "fp32"   # tcgen05 / TMA kernels for the GEMM-shaped and depthwise layers
        self.wgrad_tc = True                # tcgen05 weight gradients (stride-1 "same" and stride-2 convolutions)
        self.stem_gemm = True               # both stems as 1x1 GEMMs on one bf16 im2col of the input
        self.dgrad_s2_tc = True             # stride-2 data gradients as four parity-class conv_tc calls
        self.attn_tc = True                 # attention GEMMs (forward and backward) on the tensor cores
        self.wgrad_overlap = True           # weight gradients on a second stream (a parallel branch of the backward graph)
        self.branch_overlap = True          # spatial-branch backward beside the attention-branch / backbone backward
        self._side: Optional[torch.cuda.Stream] = None
        self._side2: Optional[torch.cuda.Stream] = None
        self._branch: Optional[Tuple[int, int, int]] = None
        self._side_used = False
        self._zero_cache: Dict[int, torch.Tensor] = {}
        self.use_graph = True               # replay the step as two CUDA graphs once its geometry has been seen
        self.graph_after = 2                # eager steps per geometry before the capture (lazy tables, attributes)
        self.max_graphs = 2                 # captured geometries kept (each pins a step's activations)
        self._gsteps: Dict[tuple, "_GraphedStep"] = {}
        self._active: Optional["_GraphedStep"] = None
        self._stems: Optional[Tuple[Map, Map, tuple]] = None   # stem output maps + input shape when x needs a gradient
        self.dx: Optional[torch.Tensor] = None                  # input gradient of the last backward (None: not needed)

    # ------------------------------------------------------------------ plumbing
    @property
    def stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def _call(self, name: str, *args):
        tr = self.trace
        if tr is not None:  # bench / profiling: bracket the call with CUDA events on the launching stream
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = getattr(self.lib, name)(*args, self.stream)
            e1.record()
            tr.append((name, self.phase, e0, e1))
        else:
            rc = getattr(self.lib, name)(*args, self.stream)
        check(rc, name)
        self.launches += 1

    def _call_tc(self, name: str, *args):
        """A tensor-core / staging entry point with 2-byte operands: the bf16 schedule calls ``name`` itself, the fp16
        schedule its ``name + '_dt'`` variant with the operand type appended."""
        if self.dt == F16:
            self._call(name + "_dt", *args, F16)
        else:
            self._call(name, *args)

    def start_trace(self):
        self.trace = []

    def stop_trace(self):
        """-> [(kernel entry point, 'fwd' | 'bwd', ms)]; synchronises."""
        torch.cuda.synchronize(self.dev)
        rows = [(n, ph, e0.elapsed_time(e1)) for n, ph, e0, e1 in self.trace]
        self.trace = None
        return rows

    def new(self, N, H, W, C, dtype=None) -> Map:
        return Map(torch.empty((N, H, W, C), dtype=dtype or self.tdt, device=self.dev), N, H, W, C, C)

    def scratch(self, M: int, C: int, nq: int) -> torch.Tensor:
        n = int(self.lib.cabinet_train_scratch_floats(int(M), int(C), int(nq)))
        return torch.empty(max(n, 1), dtype=torch.float32, device=self.dev)

    def pgrad(self, p: torch.nn.Parameter) -> torch.Tensor:
        """fp32 gradient accumulator of a parameter (zeroed on first use in a backward)."""
        g = self.pgrads.get(id(p))
        if g is None:
            self._ensure_pflat()
            off, n = self._pslots[id(p)]
            g = self.pgrads[id(p)] = self._pflat[off:off + n].view(p.shape)
        return g

    @contextlib.contextmanager
    def _wgrad_stream(self):
        """Weight gradients feed nothing but the parameter gradients, so they leave the dy -> dx chain: the block runs on
        a side stream that waits for everything queued so far (dy is complete) and is joined at the end of ``backward``.
        Inside a captured backward the fork / join become parallel branches of the graph: the small layers' weight
        gradients (16-30 us kernels on a fraction of the SMs) run under the data-gradient chain.  Tensors allocated inside
        the block belong to the side stream's pool; dy / x / the flat parameter-gradient buffer live until the join."""
        if not self.wgrad_overlap or self.trace is not None or torch.device(self.dev).type != "cuda":
            yield
            return
        if self._side is None:
            self._side = torch.cuda.Stream(self.dev)
        self._side.wait_stream(torch.cuda.current_stream(self.dev))
        self._side_used = True
        with torch.cuda.stream(self._side):
            yield

    def _ensure_pflat(self):
        if self._pflat is None:  # one buffer, one fill kernel per backward instead of one per parameter
            off = 0
            self._pslots = {}
            for q in self.model.parameters():
                if not q.requires_grad:
                    continue  # frozen: no slot, no gradient
                self._pslots[id(q)] = (off, q.numel())
                off += -(-q.numel() // 64) * 64  # 256-byte aligned slots
            self._pflat = torch.zeros(max(off, 1), dtype=torch.float32, device=self.dev)

    @staticmethod
    def _dt(t: torch.Tensor) -> int:
        return dtype_code(t.dtype)

    # ------------------------------------------------------------------ ops (forward + tape entry)
    def _zeros(self, n: int) -> torch.Tensor:
        z = self._zero_cache.get(n)
        if z is None:
            z = self._zero_cache[n] = torch.zeros(n, dtype=torch.float32, device=self.dev)
        return z

    @staticmethod
    def _tc_ok(m: Map) -> bool:
        return m.dt in (BF16, F16) and m.ld % 8 == 0 and m.off % 8 == 0 and m.t.data_ptr() % 16 == 0

    def conv(self, x: Optional[Map], conv, out: Optional[Map] = None, out_dtype=None,
             nchw: Optional[torch.Tensor] = None) -> Map:
        """nn.Conv2d (bias optional) on an NHWC map or the fp32 NCHW network input.  bf16 / fp16 mode: forward and the stride-1
        data gradient run on the tensor cores (cabinet_conv_tc; the data gradient of a stride-1 convolution is the
        convolution of dy with the transposed, mirrored weights); fp32 mode and the remaining cases: CUDA-core kernels.
        The backward computes the gradient of each parameter that requires grad, and the data gradient only when the
        input map needs one.  The network input's gradient is cabinet_stem_dgrad's (``backward``): a stem on it keeps its
        output gradient when the input requires grad."""
        w, b = conv.weight, conv.bias
        w_rg, b_rg = w.requires_grad, b is not None and b.requires_grad
        need_dx = nchw is None and x.needs_grad
        cout, cin, kh, kw = w.shape
        taps = kh * kw
        stride, pad = conv.stride[0], conv.padding[0]
        if nchw is not None:
            N, _, H, W = nchw.shape
            xptr, xdt, strides = nchw.data_ptr(), F32, (3 * H * W, W, 1, H * W)
        else:
            N, H, W = x.N, x.H, x.W
            xptr, xdt, strides = x.ptr, x.dt, (H * W * x.ld, W * x.ld, x.ld, 1)
            assert x.C == cin, (x.C, cin)
        OH, OW = _out_size(H, kh, stride, pad), _out_size(W, kw, stride, pad)
        if out is None:
            out = self.new(N, OH, OW, cout, out_dtype)
        bias = b.detach() if b is not None else None
        tc = (self.use_tc and nchw is None and self._tc_ok(x) and stride in (1, 2) and (stride == 1 or (H >= 2 and W >= 2))
              and (out.dt == F32 or self._tc_ok(out)))
        if tc:
            r16, k64 = -(-cout // 16) * 16, -(-cin // 64) * 64
            wp = torch.empty((r16, taps, k64), dtype=self.tdt, device=self.dev)
            self._call("cabinet_pack_conv_weight", w.data_ptr(), cout, cin, kh, kw, wp.data_ptr(), self.dt, r16, k64, 0)
            self._call_tc("cabinet_conv_tc", x.ptr, x.ld, N, H, W, cin, wp.data_ptr(), cout, kh, kw, stride, pad,
                          (bias if bias is not None else self._zeros(cout)).data_ptr(), None, 0, out.ptr, out.dt, out.ld, OH, OW,
                          ACT_NONE)
            wdt, w_sco, w_stap = self.dt, taps * k64, k64
        else:
            wp = torch.empty((cout, taps, cin), dtype=torch.float32, device=self.dev)
            self._call("cabinet_pack_conv_weight", w.data_ptr(), cout, cin, kh, kw, wp.data_ptr(), F32, cout, cin, 0)
            self._call("cabinet_conv2d_simt", xptr, xdt, *strides, 0, wp.data_ptr(), F32, taps * cin, 1, 0,
                       bias.data_ptr() if bias is not None else None, None, 0, out.ptr, out.dt, out.ld, 0, 1, N, H, W, cin,
                       cout, kh, kw, stride, pad, OH, OW, ACT_NONE, 1.0)
            wdt, w_sco, w_stap = F32, taps * cin, cin
        out.needs_grad = need_dx or w_rg or b_rg or (nchw is not None and self._stems is not None)

        def backward(g: _Grads):
            dy = g.get(out) if out.needs_grad else None
            if dy is None:
                return
            if w_rg or b_rg:
                with self._wgrad_stream():
                    if b_rg:
                        sc = self.scratch(N * OH * OW, cout, 1)
                        self._call("cabinet_col_sum", dy.ptr, dy.ld, dy.dt, N * OH * OW, cout, self.pgrad(b).data_ptr(), 1,
                                   sc.data_ptr())
                    if w_rg and (self.use_tc and self.wgrad_tc and nchw is None and kh == kw and self._tc_ok(x)
                                 and self._tc_ok(dy)
                                 and ((stride == 1 and 2 * pad == kh - 1) or (stride == 2 and H >= 2 and W >= 2))):
                        n = int(self.lib.cabinet_conv_wgrad_tc_scratch_floats(N, H, W, cin, cout, kh, kw, stride, pad))
                        sc = torch.empty(n, dtype=torch.float32, device=self.dev)
                        self._call_tc("cabinet_conv_wgrad_tc", dy.ptr, dy.ld, x.ptr, x.ld, self.pgrad(w).data_ptr(), N, H, W,
                                      cin, cout, kh, kw, stride, pad, sc.data_ptr())
                    elif w_rg:
                        n = int(self.lib.cabinet_conv_wgrad_scratch_floats(N, OH, OW, cin, cout, kh, kw))
                        sc = torch.empty(n, dtype=torch.float32, device=self.dev)
                        self._call("cabinet_conv_wgrad", dy.ptr, dy.ld, dy.dt, xptr, xdt, *strides, self.pgrad(w).data_ptr(),
                                   N, H, W, cin, cout, kh, kw, stride, pad, OH, OW, sc.data_ptr())
            if not need_dx:
                return
            if dy.dt != x.dt:  # fp32 class-logit gradients into a 2-byte activation gradient (pixel stride padded to 8)
                dyc = Map(torch.empty((N, OH, OW, -(-cout // 8) * 8), dtype=x.t.dtype, device=self.dev), N, OH, OW, cout,
                          -(-cout // 8) * 8)
                self._call("cabinet_affine_act", dy.ptr, dy.ld, dy.dt, None, None, None, 0.0, None, 0, dyc.ptr, dyc.ld,
                           dyc.dt, N * OH * OW, OH * OW, cout, ACT_NONE)
                dy = dyc
            dx, acc = g.out(x)
            if self.use_tc and stride == 1 and self._tc_ok(dy) and self._tc_ok(dx) and (OH, OW) == (H, W):
                r16, k64 = -(-cin // 16) * 16, -(-cout // 64) * 64
                wt = torch.empty((r16, taps, k64), dtype=self.tdt, device=self.dev)
                self._call("cabinet_pack_conv_weight", w.data_ptr(), cout, cin, kh, kw, wt.data_ptr(), self.dt, r16, k64, 1)
                self._call_tc("cabinet_conv_tc", dy.ptr, dy.ld, N, H, W, cout, wt.data_ptr(), cin, kh, kw, 1, kh - 1 - pad,
                              self._zeros(cin).data_ptr(), dx.ptr if acc else None, dx.ld if acc else 0, dx.ptr, dx.dt, dx.ld,
                              H, W, ACT_NONE)
                return
            if (self.use_tc and self.dgrad_s2_tc and stride == 2 and kh == kw and not acc and self._tc_ok(dy)
                    and self._tc_ok(dx) and H >= 2 and W >= 2 and self._parity_pads(kh, pad) is not None):
                # stride 2: four input-parity classes, each the stride-1 convolution of dy with a sub-filter, written
                # through a strided view of dx (cabinet_conv_tc_view)
                r16, k64 = -(-cin // 16) * 16, -(-cout // 64) * 64
                for py in range(2):
                    for px in range(2):
                        (kh2, pad2), (kw2, padx2) = self._parity_geom(kh, pad, py), self._parity_geom(kw, pad, px)
                        hc, wc = (H - py + 1) // 2, (W - px + 1) // 2
                        if hc == 0 or wc == 0:
                            continue
                        wt = torch.empty((r16, kh2 * kw2, k64), dtype=self.tdt, device=self.dev)
                        self._call_tc("cabinet_pack_conv_weight_parity", w.data_ptr(), cout, cin, kh, pad, py, px, kh2, kw2,
                                      pad2, wt.data_ptr(), r16, k64)
                        view = dx.ptr + (py * W + px) * dx.ld * 2
                        self._call_tc("cabinet_conv_tc_view", dy.ptr, dy.ld, N, OH, OW, cout, wt.data_ptr(), cin, kh2, kw2,
                                      pad2, self._zeros(cin).data_ptr(), view, dx.ld, hc, wc, 2, 2 * W, H * W)
                return
            self._call("cabinet_conv_dgrad", dy.ptr, dy.ld, dy.dt, wp.data_ptr(), wdt, w_sco, w_stap, dx.ptr, dx.ld, N, H, W,
                       cin, cout, kh, kw, stride, pad, OH, OW, acc)

        self.tape.append(backward)
        return out

    @staticmethod
    def _parity_geom(k: int, pad: int, par: int):
        """(taps, pad) of the stride-1 sub-convolution that yields the input rows of parity ``par`` of a stride-2
        convolution's data gradient: row 2a + par meets ky = par + pad - 2 off, off = dy row - a."""
        offs = [(par + pad - ky) // 2 for ky in range(k) if (par + pad - ky) % 2 == 0]
        if not offs:
            return 1, 0   # no tap of this parity: a 1-tap sub-filter of zeros
        return max(offs) - min(offs) + 1, -min(offs)

    @classmethod
    def _parity_pads(cls, k: int, pad: int):
        """cabinet_conv_tc takes ONE padding for both axes: usable when both parities need the same one (3x3 / pad 1 and
        7x7 / pad 3 do; 5x5 / pad 2 does not) -> that padding, else None."""
        p0, p1 = cls._parity_geom(k, pad, 0)[1], cls._parity_geom(k, pad, 1)[1]
        return p0 if p0 == p1 else None

    # im2col footprint of CABiNet's stems: 3 x 7 x 7 = 147 columns (a standalone MobileNetV3 uses its stem's 3 x 3 x 3)
    STEM_K = 7

    @staticmethod
    def stem_ld(k: int) -> int:
        """Pixel stride of the im2col over a k x k footprint: 3 k^2 columns padded to 8 (7: 152, 3: 32)."""
        return -(-3 * k * k // 8) * 8

    def stem_im2col(self, x: torch.Tensor, k: int = STEM_K) -> Map:
        """2-byte (bf16 / fp16) im2col [N, H/2, W/2, stem_ld(k)] of the fp32 NCHW input over the k x k / stride-2 /
        pad-(k-1)/2 footprint.  CABiNet's 7x7 one is shared by both stem convolutions (the 3x3 / pad-1 backbone stem is
        its centre): read once, used by two forward GEMMs and two weight-gradient GEMMs on the tensor cores."""
        N, _, H, W = x.shape
        pad, ld = (k - 1) // 2, self.stem_ld(k)
        OH, OW = _out_size(H, k, 2, pad), _out_size(W, k, 2, pad)
        xcol = Map(torch.empty((N, OH, OW, ld), dtype=self.tdt, device=self.dev), N, OH, OW, ld, ld)
        self._call_tc("cabinet_im2col_nchw", x.data_ptr(), N, 3, H, W, k, 2, pad, xcol.ptr, xcol.ld)
        return xcol

    def conv_stem(self, xcol: Map, conv, K: int = STEM_K) -> Map:
        """A stem convolution (7x7 s2 p3, or 3x3 s2 p1 embedded in the same footprint) as a 1x1 GEMM on the im2col matrix
        of the K x K footprint."""
        w = conv.weight
        cout, cin, k, _ = w.shape
        assert cin == 3 and conv.stride[0] == 2 and (k, conv.padding[0]) in ((7, 3), (3, 1)) and conv.bias is None
        assert k <= K and xcol.ld == self.stem_ld(K)
        N, OH, OW, LD = xcol.N, xcol.H, xcol.W, xcol.ld
        out = self.new(N, OH, OW, cout)
        r16, k64 = -(-cout // 16) * 16, -(-LD // 64) * 64
        wbig = torch.zeros((cout, LD), dtype=torch.float32, device=self.dev)
        self.launches += 1
        wp = torch.empty((r16, 1, k64), dtype=self.tdt, device=self.dev)
        self._call("cabinet_embed_filter", w.data_ptr(), cout, 3, k, K, wbig.data_ptr(), LD, 0)
        self._call("cabinet_pack_conv_weight", wbig.data_ptr(), cout, LD, 1, 1, wp.data_ptr(), self.dt, r16, k64, 0)
        self._call_tc("cabinet_conv_tc", xcol.ptr, xcol.ld, N, OH, OW, LD, wp.data_ptr(), cout, 1, 1, 1, 0,
                      self._zeros(cout).data_ptr(), None, 0, out.ptr, out.dt, out.ld, OH, OW, ACT_NONE)
        out.needs_grad = w.requires_grad or self._stems is not None  # the input's gradient: cabinet_stem_dgrad

        def backward(g: _Grads):
            dy = g.get(out) if out.needs_grad and w.requires_grad else None
            if dy is None:
                return
            with self._wgrad_stream():
                dwbig = torch.zeros((cout, LD), dtype=torch.float32, device=self.dev)
                self.launches += 1
                n = int(self.lib.cabinet_conv_wgrad_tc_scratch_floats(N, OH, OW, LD, cout, 1, 1, 1, 0))
                sc = torch.empty(n, dtype=torch.float32, device=self.dev)
                self._call_tc("cabinet_conv_wgrad_tc", dy.ptr, dy.ld, xcol.ptr, xcol.ld, dwbig.data_ptr(), N, OH, OW, LD, cout,
                              1, 1, 1, 0, sc.data_ptr())
                self._call("cabinet_embed_filter", self.pgrad(w).data_ptr(), cout, 3, k, K, dwbig.data_ptr(), LD, 1)

        self.tape.append(backward)
        return out

    def dwconv(self, x: Map, conv) -> Map:
        """Depthwise nn.Conv2d (groups = C, no bias).  bf16 / fp16 mode: the TMA-staged kernel forward, and for stride 1 also
        backward (the data gradient is the depthwise convolution of dy with the mirrored filter)."""
        w = conv.weight
        C, k, stride = w.shape[0], w.shape[2], conv.stride[0]
        p = (k - 1) // 2
        OH, OW = _out_size(x.H, k, stride, p), _out_size(x.W, k, stride, p)
        out = self.new(x.N, OH, OW, C)
        wp = torch.empty((k * k, C), dtype=torch.float32, device=self.dev)
        self._call("cabinet_pack_dw_weight", w.data_ptr(), C, k, 0, wp.data_ptr())
        tma = self.use_tc and self._tc_ok(x) and self._tc_ok(out) and C % 8 == 0
        if tma:
            self._call_tc("cabinet_dwconv_tma", x.ptr, x.ld, wp.data_ptr(), self._zeros(C).data_ptr(), out.ptr, out.ld, x.N,
                          x.H, x.W, C, k, stride, OH, OW, ACT_NONE, None)
        else:
            self._call("cabinet_dwconv", x.ptr, x.ld, wp.data_ptr(), self._zeros(C).data_ptr(), out.ptr, out.ld, x.dt, x.N, x.H,
                       x.W, C, k, stride, OH, OW, ACT_NONE, None)

        w_rg = w.requires_grad
        out.needs_grad = x.needs_grad or w_rg

        def backward(g: _Grads):
            dy = g.get(out) if out.needs_grad else None
            if dy is None:
                return
            if w_rg:
                with self._wgrad_stream():
                    sc = self.scratch(x.N * OH * OW, C, k * k)
                    self._call("cabinet_dwconv_wgrad", dy.ptr, dy.ld, x.ptr, x.ld, x.dt, self.pgrad(w).data_ptr(), x.N, x.H,
                               x.W, C, k, stride, OH, OW, sc.data_ptr())
            if not x.needs_grad:
                return
            dx, acc = g.out(x)
            if tma and stride == 1 and self._tc_ok(dy):
                wf = torch.empty((k * k, C), dtype=torch.float32, device=self.dev)
                self._call("cabinet_pack_dw_weight", w.data_ptr(), C, k, 1, wf.data_ptr())
                tgt = self.new(x.N, x.H, x.W, C) if acc else dx
                self._call_tc("cabinet_dwconv_tma", dy.ptr, dy.ld, wf.data_ptr(), self._zeros(C).data_ptr(), tgt.ptr, tgt.ld,
                              x.N, x.H, x.W, C, k, 1, x.H, x.W, ACT_NONE, None)
                if acc:
                    self._call("cabinet_add", dx.ptr, dx.ld, tgt.ptr, tgt.ld, dx.ptr, dx.ld, dx.dt, x.N * x.H * x.W, C)
                return
            self._call("cabinet_dwconv_dgrad", dy.ptr, dy.ld, dy.dt, wp.data_ptr(), dx.ptr, dx.ld, x.N, x.H, x.W, C, k, stride,
                       OH, OW, acc)

        self.tape.append(backward)
        return out

    def bn(self, z: Map, bn, act: int, res: Optional[Map] = None, out: Optional[Map] = None) -> Map:
        """BatchNorm2d (+activation) (+ residual add), per module as PyTorch does it: a module in training mode normalises
        with the batch statistics and updates its running statistics; one in eval mode (``bn.eval()`` inside a
        ``.train()`` model) normalises with its running statistics and leaves them, and ``num_batches_tracked``, alone."""
        M, C = z.N * z.H * z.W, z.C
        stats = torch.empty((4, C), dtype=torch.float32, device=self.dev)
        frozen = not bn.training
        if frozen:
            self._call("cabinet_bn_frozen_stats", bn.weight.data_ptr(), bn.bias.data_ptr(), bn.running_mean.data_ptr(),
                       bn.running_var.data_ptr(), float(bn.eps), C, stats.data_ptr())
        else:
            sc = self.scratch(M, C, 2)
            self._call("cabinet_bn_train_stats", z.ptr, z.ld, z.dt, M, C, bn.weight.data_ptr(), bn.bias.data_ptr(),
                       float(bn.eps), BN_MOMENTUM if bn.momentum is None else float(bn.momentum),
                       bn.running_mean.data_ptr(), bn.running_var.data_ptr(), stats.data_ptr(), sc.data_ptr())
            self._bn_seen.append(bn.num_batches_tracked)  # += 1 for all of them at the end of the forward (one kernel)
        if out is None:
            out = self.new(z.N, z.H, z.W, C)
        self._call("cabinet_affine_act", z.ptr, z.ld, z.dt, stats[2].data_ptr(), stats[3].data_ptr(), None, 0.0,
                   res.ptr if res is not None else None, res.ld if res is not None else 0, out.ptr, out.ld, out.dt, M,
                   z.H * z.W, C, act)
        g_rg, b_rg = bn.weight.requires_grad, bn.bias.requires_grad
        res_rg = res is not None and res.needs_grad
        out.needs_grad = z.needs_grad or g_rg or b_rg or res_rg

        def backward(g: _Grads):
            dy = g.get(out) if out.needs_grad else None
            if dy is None:
                return
            if res_rg:  # identity branch: d res += dy
                self.add_grad(g, res, dy)
            dgamma = self.pgrad(bn.weight).data_ptr() if g_rg else None
            dbeta = self.pgrad(bn.bias).data_ptr() if b_rg else None
            if z.needs_grad and not frozen:
                dz, acc = g.out(z)
                sc2 = self.scratch(M, C, 4)
                self._call("cabinet_bn_train_backward", dy.ptr, dy.ld, z.ptr, z.ld, z.dt, stats.data_ptr(), act, dgamma, dbeta,
                           dz.ptr, dz.ld, M, C, acc, sc2.data_ptr())
            elif z.needs_grad or g_rg or b_rg:
                # eval mode: dz = scale * g in the same pass as the reductions; or a training module whose input needs no
                # gradient: its dgamma / dbeta are the same two sums over the batch statistics
                dz, acc = g.out(z) if z.needs_grad else (None, 0)
                sc2 = self.scratch(M, C, 2) if (g_rg or b_rg) else None
                self._call("cabinet_bn_frozen_backward", dy.ptr, dy.ld, z.ptr, z.ld, z.dt, stats.data_ptr(), act, dgamma,
                           dbeta, dz.ptr if dz is not None else None, dz.ld if dz is not None else 0, M, C, acc,
                           sc2.data_ptr() if sc2 is not None else None)

        self.tape.append(backward)
        return out

    def add_grad(self, g: _Grads, target: Map, dy: Map):
        """grad(target) += dy (or = dy for the first writer)."""
        dt, acc = g.out(target)
        M = target.N * target.H * target.W
        if acc:
            self._call("cabinet_add", dt.ptr, dt.ld, dy.ptr, dy.ld, dt.ptr, dt.ld, dt.dt, M, target.C)
        else:
            self._call("cabinet_affine_act", dy.ptr, dy.ld, dy.dt, None, None, None, 0.0, None, 0, dt.ptr, dt.ld, dt.dt, M,
                       target.H * target.W, target.C, ACT_NONE)

    def channel_mean_sum(self, v: Map) -> torch.Tensor:
        """[N][C] fp32 sums over the pixels of every image (deterministic two-level sum)."""
        out = torch.empty((v.N, v.C), dtype=torch.float32, device=self.dev)
        scratch = torch.zeros(128 + v.N * 64 * v.C, dtype=torch.float32, device=self.dev)
        self.launches += 1
        self._call("cabinet_channel_sum", v.ptr, v.ld, v.dt, v.N, v.H * v.W, v.C, out.data_ptr(), scratch.data_ptr(),
                   scratch.numel() * 4)
        return out

    def gate(self, v: Map, w1, b1, w2, b2, gate_act: int, act: int, plus: float, out: Optional[Map] = None) -> Map:
        """y = act(v * (s + plus)), s = gate(W2 relu(W1 mean(v) + b1) + b2): SELayer (mobilenetv3.py:68-83) followed by the
        block activation, or the FFM attention (cabinet.py:146-153, plus = 1)."""
        N, C, HW = v.N, v.C, v.H * v.W
        J = w1.shape[0]
        sums = self.channel_mean_sum(v)
        hidden = torch.empty((N, J), dtype=torch.float32, device=self.dev)
        s = torch.empty((N, C), dtype=torch.float32, device=self.dev)
        w1f, w2f = w1.detach().reshape(J, C), w2.detach().reshape(C, J)
        self._call("cabinet_gate_fc", sums.data_ptr(), 1.0 / HW, w1f.data_ptr(), b1.data_ptr() if b1 is not None else None,
                   hidden.data_ptr(), N, C, J, ACT_RELU, 0)
        self._call("cabinet_gate_fc", hidden.data_ptr(), 1.0, w2f.data_ptr(), b2.data_ptr() if b2 is not None else None,
                   s.data_ptr(), N, J, C, gate_act, 0)
        if out is None:
            out = self.new(v.N, v.H, v.W, C)
        self._call("cabinet_affine_act", v.ptr, v.ld, v.dt, None, None, s.data_ptr(), plus, None, 0, out.ptr, out.ld, out.dt,
                   N * HW, HW, C, act)
        rg = [p is not None and p.requires_grad for p in (w1, b1, w2, b2)]
        out.needs_grad = v.needs_grad or any(rg)

        def backward(g: _Grads):
            dy = g.get(out) if out.needs_grad else None
            if dy is None:
                return
            ds = torch.empty((N, C), dtype=torch.float32, device=self.dev)
            sc = torch.empty(N * int(self.lib.cabinet_train_scratch_floats(HW, C, 1)), dtype=torch.float32, device=self.dev)
            self._call("cabinet_gate_scale_backward", dy.ptr, dy.ld, v.ptr, v.ld, v.dt, s.data_ptr(), plus, act, ds.data_ptr(), N,
                       HW, C, sc.data_ptr())
            dm = torch.empty((N, C), dtype=torch.float32, device=self.dev)
            sc2 = torch.empty(N * (C + J), dtype=torch.float32, device=self.dev)
            # the kernel writes both weight gradients on its way to dm: a frozen weight's goes to a scratch buffer
            dw = [self.pgrad(p) if r else None for p, r in zip((w1, b1, w2, b2), rg)]
            for i in (0, 2):
                if dw[i] is None:
                    dw[i] = torch.empty(J * C, dtype=torch.float32, device=self.dev)
            self._call("cabinet_gate_mlp_backward", sums.data_ptr(), 1.0 / HW, w1f.data_ptr(), w2f.data_ptr(), hidden.data_ptr(),
                       s.data_ptr(), ds.data_ptr(), gate_act, N, C, J, *(t.data_ptr() if t is not None else None for t in dw),
                       dm.data_ptr(), sc2.data_ptr())
            if not v.needs_grad:
                return
            dv, acc = g.out(v)
            self._call("cabinet_gate_apply_backward", dy.ptr, dy.ld, v.ptr, v.ld, v.dt, s.data_ptr(), plus, dm.data_ptr(), 1.0 / HW,
                       act, dv.ptr, dv.ld, N, HW, C, acc)

        self.tape.append(backward)
        return out

    def _resample_call(self, src: Map, dst: Map, ty, tx, flags: int):
        self._call("cabinet_resample_sep", src.ptr, src.dt, src.H * src.W * src.ld, src.W * src.ld, src.ld, 1, dst.ptr, dst.dt,
                   dst.H * dst.W * dst.ld, dst.W * dst.ld, dst.ld, 1, src.N, dst.H, dst.W, src.C,
                   *(t.data_ptr() for t in ty), *(t.data_ptr() for t in tx), flags)

    def _reduce_two_pass(self, src: Map, dst: Map, ty, tx, acc: int):
        """A reducing operator with >= 64 taps per output (a pool to 1 x 1 or 3 x 3, the adjoint of the up-sampling of such
        a map) as two separable passes, first along x, then along y: 32 + 32 taps per output instead of 1024 gathered by
        one thread (0.22 -> ~0.03 ms for the 1 x 1 PSP bin)."""
        tmp = self.new(src.N, src.H, dst.W, src.C, torch.float32)
        self._resample_call(src, tmp, self.tables.get("identity", src.H, src.H, False), tx, 0)
        self._resample_call(tmp, dst, ty, self.tables.get("identity", dst.W, dst.W, False), acc)

    def resample(self, src: Map, kind: str, OH: int, OW: int, out: Optional[Map] = None, out_dtype=None) -> Map:
        """Bilinear resize (align_corners=False) or adaptive average pool of an NHWC map, + its adjoint on the tape."""
        if out is None:
            out = self.new(src.N, OH, OW, src.C, out_dtype or src.t.dtype)
        ty, tx = self.tables.get(kind, src.H, OH, False), self.tables.get(kind, src.W, OW, False)
        up = OH * OW >= src.H * src.W  # an upsample reads <= 2 x 2 taps per output, its adjoint many (and vice versa for a pool)
        many = max(src.H * src.W, OH * OW) >= 64 * min(src.H * src.W, OH * OW)  # >= 64 taps per output on the reducing side
        if many and not up:
            self._reduce_two_pass(src, out, ty, tx, 0)
        else:
            self._resample_call(src, out, ty, tx, 4 if up else 0)  # bit 2: few taps per output -> vector kernel
        out.needs_grad = src.needs_grad

        def backward(g: _Grads):
            dy = g.get(out) if out.needs_grad else None
            if dy is None:
                return
            dx, acc = g.out(src)
            ay, ax = self.tables.get(kind, src.H, OH, True), self.tables.get(kind, src.W, OW, True)
            dym = Map(dy.t, dy.N, OH, OW, dy.C, dy.ld, dy.off)
            dxm = Map(dx.t, dx.N, src.H, src.W, dx.C, dx.ld, dx.off)
            if many and up:
                self._reduce_two_pass(dym, dxm, ay, ax, acc)
            else:
                self._resample_call(dym, dxm, ay, ax, acc | (0 if up else 4))

        self.tape.append(backward)
        return out

    def psp(self, x: Map, project) -> Map:
        """PSPModule (cab.py:46-76): cat[x, up(pool_s(x)) for s in (1,3,6,8)] -> 1x1 project."""
        cat = self.new(x.N, x.H, x.W, 5 * x.C)
        ident = cat.slice(0, x.C)
        self._call("cabinet_affine_act", x.ptr, x.ld, x.dt, None, None, None, 0.0, None, 0, ident.ptr, ident.ld, ident.dt,
                   x.N * x.H * x.W, x.H * x.W, x.C, ACT_NONE)
        cat.needs_grad = ident.needs_grad = x.needs_grad  # every slice of the concatenation is a function of x alone

        def ident_bwd(g: _Grads):
            dy = g.get(ident) if ident.needs_grad else None
            if dy is not None:
                self.add_grad(g, x, dy)

        self.tape.append(ident_bwd)
        for i, s in enumerate(PSP_SIZES):
            pooled = self.resample(x, "pool", s, s)
            self.resample(pooled, "bilinear", x.H, x.W, out=cat.slice((i + 1) * x.C, x.C))
        return self.conv(cat, project)

    def attention(self, q: Map, k: Map, v: Map) -> Map:
        """softmax(q k^T / sqrt(d)) v per image with the probabilities kept for the backward (cab.py:149-153).  q, k: [N, L, d]
        (d = key width, which sets the scale), v: [N, L, dv]; -> ctx [N, L, dv]."""
        N, L, d, dv = q.N, q.H * q.W, q.C, v.C
        alpha = float(d) ** -0.5
        if (self.use_tc and self.attn_tc and L % 128 == 0 and d % 64 == 0 and dv % 64 == 0
                and all(self._tc_ok(t) and t.ld == t.C for t in (q, k, v))):
            return self._attention_tc(q, k, v, alpha)
        s = torch.empty((N, L, L), dtype=torch.float32, device=self.dev)
        p = torch.empty((N, L, L), dtype=torch.float32, device=self.dev)
        ctx = self.new(q.N, q.H, q.W, dv)

        def gemm(xp, xdt, sxw, sxc, xbs, wpt, wdt, w_sco, w_sk, wbs, yp, ydt, ldy, ybs, Mr, Kd, Nc, al=1.0):
            # out[b][m][co] = al * sum_k x[b][m][k] w[b][co][k]
            self._call("cabinet_conv2d_simt", xp, xdt, 0, 0, sxw, sxc, xbs, wpt, wdt, w_sco, w_sk, wbs, None, None, 0, yp, ydt,
                       ldy, ybs, N, 1, 1, Mr, Kd, Nc, 1, 1, 1, 0, 1, Mr, ACT_NONE, al)

        gemm(q.ptr, q.dt, q.ld, 1, L * q.ld, k.ptr, k.dt, k.ld, 1, L * k.ld, s.data_ptr(), F32, L, L * L, L, d, L, alpha)
        self._call("cabinet_softmax_rows", s.data_ptr(), p.data_ptr(), F32, N * L, L)
        gemm(p.data_ptr(), F32, L, 1, L * L, v.ptr, v.dt, 1, v.ld, L * v.ld, ctx.ptr, ctx.dt, ctx.ld, L * ctx.ld, L, L, dv)
        ctx.needs_grad = q.needs_grad or k.needs_grad or v.needs_grad

        def backward(g: _Grads):
            do = g.get(ctx) if ctx.needs_grad else None
            if do is None:
                return
            dp = s  # the raw scores are not needed any more: reuse their buffer
            ds = torch.empty((N, L, L), dtype=torch.float32, device=self.dev)
            dq, dk = (self.new(q.N, q.H, q.W, d) for _ in range(2))
            dV = self.new(q.N, q.H, q.W, dv)
            # dV[j][c] = sum_i P[i][j] dO[i][c]
            gemm(p.data_ptr(), F32, 1, L, L * L, do.ptr, do.dt, 1, do.ld, L * do.ld, dV.ptr, dV.dt, dv, L * dv, L, L, dv)
            # dP[i][j] = sum_c dO[i][c] V[j][c]
            gemm(do.ptr, do.dt, do.ld, 1, L * do.ld, v.ptr, v.dt, v.ld, 1, L * v.ld, dp.data_ptr(), F32, L, L * L, L, dv, L)
            self._call("cabinet_softmax_backward", p.data_ptr(), dp.data_ptr(), ds.data_ptr(), N * L, L, alpha)
            # dQ[i][c] = sum_j dS[i][j] K[j][c];  dK[j][c] = sum_i dS[i][j] Q[i][c]
            gemm(ds.data_ptr(), F32, L, 1, L * L, k.ptr, k.dt, 1, k.ld, L * k.ld, dq.ptr, dq.dt, d, L * d, L, L, d)
            gemm(ds.data_ptr(), F32, 1, L, L * L, q.ptr, q.dt, 1, q.ld, L * q.ld, dk.ptr, dk.dt, d, L * d, L, L, d)
            for tgt, src in ((q, dq), (k, dk), (v, dV)):
                if tgt.needs_grad:
                    self.add_grad(g, tgt, src)

        self.tape.append(backward)
        return ctx

    def _attention_tc(self, q: Map, k: Map, v: Map, alpha: float) -> Map:
        """The same attention with all six GEMMs on the tensor cores (bf16 / fp16 operands, fp32 accumulation): a dense [L][d] map
        of an image IS a cabinet_conv_tc weight matrix (rows = tokens, k = channels), so S = Q K^T and dP = dO V^T are 1x1
        convolutions with per-image weights K / V, P V and dQ = dS K the same with K^T / V^T ([d][L], one small transpose
        each), and dV = P^T dO, dK = dS^T Q reduce over the token ("pixel") index: the weight-gradient GEMM, batched per image."""
        N, L, d, dv, H, W = q.N, q.H * q.W, q.C, v.C, q.H, q.W
        dev, bf = self.dev, self.tdt
        s = torch.empty((N, L, L), dtype=torch.float32, device=dev)
        p = torch.empty((N, L, L), dtype=torch.float32, device=dev)
        p16 = torch.empty((N, L, L), dtype=bf, device=dev)
        vt = torch.empty((N, dv, L), dtype=bf, device=dev)
        ctx = self.new(N, H, W, dv)
        zL, zd, zv = self._zeros(L), self._zeros(d), self._zeros(dv)

        def gemm(x_ptr, ldx, cin, w_ptr, cout, bias, y_ptr, ydt, ldy):
            # y[n][l][co] = sum_k x[n][l][k] w[n][co][k]   (w: [N][cout][cin] 2-byte, dense)
            self._call_tc("cabinet_conv_tc_imgw", x_ptr, ldx, N, H, W, cin, w_ptr, cout * cin, cout, 1, 1, 1, 0,
                          bias.data_ptr(), None, 0, y_ptr, ydt, ldy, H, W, ACT_NONE)

        gemm(q.ptr, q.ld, d, k.ptr, L, zL, s.data_ptr(), F32, L)
        self._call_tc("cabinet_attn_softmax", s.data_ptr(), alpha, p.data_ptr(), p16.data_ptr(), N * L, L)
        self._call_tc("cabinet_transpose_tokens", v.ptr, v.ld, vt.data_ptr(), N, L, dv)
        gemm(p16.data_ptr(), L, L, vt.data_ptr(), dv, zv, ctx.ptr, ctx.dt, ctx.ld)
        ctx.needs_grad = q.needs_grad or k.needs_grad or v.needs_grad

        def backward(g: _Grads):
            do = g.get(ctx) if ctx.needs_grad else None
            if do is None:
                return
            dp = s  # the raw scores are not needed any more: reuse their buffer
            ds16 = torch.empty((N, L, L), dtype=bf, device=dev)
            kt = torch.empty((N, d, L), dtype=bf, device=dev)
            dq = self.new(N, H, W, d)
            dk32 = torch.empty((N, L, d), dtype=torch.float32, device=dev)
            dv32 = torch.empty((N, L, dv), dtype=torch.float32, device=dev)

            def wgrad(a, x_map, out):  # out[n][j][c] = sum_i a[n][i][j] x[n][i][c]
                self._call_tc("cabinet_conv_wgrad_tc_batched", a.data_ptr(), L, x_map.ptr, x_map.ld, out.data_ptr(), N, H, W,
                              x_map.C, L)

            wgrad(p16, do, dv32)                                                  # dV[j][c] = sum_i P[i][j] dO[i][c]
            gemm(do.ptr, do.ld, dv, v.ptr, L, zL, dp.data_ptr(), F32, L)          # dP[i][j] = sum_c dO[i][c] V[j][c]
            self._call_tc("cabinet_attn_softmax_backward", p.data_ptr(), dp.data_ptr(), ds16.data_ptr(), N * L, L, alpha)
            self._call_tc("cabinet_transpose_tokens", k.ptr, k.ld, kt.data_ptr(), N, L, d)
            gemm(ds16.data_ptr(), L, L, kt.data_ptr(), d, zd, dq.ptr, dq.dt, dq.ld)  # dQ[i][c] = sum_j dS[i][j] K[j][c]
            wgrad(ds16, q, dk32)                                                  # dK[j][c] = sum_i dS[i][j] Q[i][c]
            dk, dV = self.new(N, H, W, d), self.new(N, H, W, dv)
            for src, dst in ((dk32, dk), (dv32, dV)):  # fp32 -> the activation dtype
                self._call("cabinet_affine_act", src.data_ptr(), dst.C, F32, None, None, None, 0.0, None, 0, dst.ptr, dst.ld,
                           dst.dt, N * L, L, dst.C, ACT_NONE)
            for tgt, src in ((q, dq), (k, dk), (v, dV)):
                if tgt.needs_grad:
                    self.add_grad(g, tgt, src)

        self.tape.append(backward)
        return ctx

    def cab(self, feat: Map, block, out: Map):
        """ContextAggregationBlock ``block``: out = gamma * global(feat) + local(feat) (cab.py:131-162,175-184,213-216)."""
        ga = block.global_attn
        q = self.bn(self.conv(feat, ga.to_query[0]), ga.to_query[1], ACT_RELU)
        k = self.psp(self.bn(self.conv(feat, ga.to_key[0]), ga.to_key[1], ACT_RELU), ga.psp_key.project)
        v = self.psp(self.conv(feat, ga.to_value), ga.psp_value.project)
        ctx = self.attention(q, k, v)
        gl = self.conv(ctx, ga.project_out)
        r = feat
        for dwb in block.local_attn.refine:
            r = self.bn(self.dwconv(r, dwb.block[0]), dwb.block[1], ACT_RELU)
        self.cab_combine(gl, feat, r, block.gamma, out)

    def cab_combine(self, gmap: Map, x: Map, r: Map, gamma, out: Map):
        """out = gamma * global + x + x * sigmoid(r) (cab.py:175-184,213-216)."""
        M = x.N * x.H * x.W
        gm = gamma.detach().float().contiguous()
        self._call("cabinet_cab_combine", gmap.ptr, x.ptr, r.ptr, out.ptr, out.ld, gm.data_ptr(), self.dt, M, x.C)
        out.needs_grad = gmap.needs_grad or x.needs_grad or r.needs_grad or gamma.requires_grad

        def backward(g: _Grads):
            dy = g.get(out) if out.needs_grad else None
            if dy is None:
                return
            # one elementwise pass writes all three data gradients and the gamma partials; the producers of the maps that
            # need no gradient skip theirs, and a frozen gamma's sum goes to a scratch slot
            dg, _ = g.out(gmap)
            dr, _ = g.out(r)
            dx, acc = g.out(x)
            sc = self.scratch(M, x.C, 1)
            dgamma = self.pgrad(gamma) if gamma.requires_grad else torch.empty(1, dtype=torch.float32, device=self.dev)
            self._call("cabinet_cab_combine_backward", dy.ptr, dy.ld, gmap.ptr, x.ptr, r.ptr, gm.data_ptr(), self.dt, dg.ptr,
                       dx.ptr, dr.ptr, dgamma.data_ptr(), M, x.C, acc, sc.data_ptr())

        self.tape.append(backward)

    def logits_up(self, src: Map, H: int, W: int, odt: torch.dtype) -> torch.Tensor:
        """x8 bilinear of the fp32 class map -> NCHW logits (cabinet.py:240-245) + its adjoint."""
        N, C = src.N, src.C
        y = torch.empty((N, C, H, W), dtype=odt, device=self.dev)
        self._call("cabinet_upsample_logits_nchw", src.ptr, N, src.H, src.W, C, y.data_ptr(), self._dt(y), H, W)

        def backward(g: _Grads, dy_nchw: torch.Tensor):
            if not src.needs_grad:
                return
            dy_nchw = dy_nchw.contiguous()
            dx, acc = g.out(src)
            ay, ax = self.tables.get("bilinear", src.H, H, True), self.tables.get("bilinear", src.W, W, True)
            self._call("cabinet_resample_sep", dy_nchw.data_ptr(), self._dt(dy_nchw), C * H * W, W, 1, H * W, dx.ptr, dx.dt,
                       src.H * src.W * dx.ld, src.W * dx.ld, dx.ld, 1, N, src.H, src.W, C, *(t.data_ptr() for t in ay),
                       *(t.data_ptr() for t in ax), acc | 2)  # bit 1: planar input, 16 x 16 taps -> row-band kernel

        return y, backward

    def mobilenet(self, f: Map, mob, out: Optional[Map] = None) -> Map:
        """The MobileNetV3 ``mob`` after its stem: the inverted-residual blocks and ``mobile.conv`` (mobilenetv3.py:102-159,
        202-205).  ``f``: the stem's output; ``out``: where ``mobile.conv`` writes (a channel slice of CABiNet's b1 concat
        buffer) or None."""
        for blk in list(mob.features)[1:]:
            s, c = blk.spec, blk.conv
            act = ACT_HSWISH if s["hs"] else ACT_RELU
            res = f if s["identity"] else None
            if s["expand"]:
                h = self.bn(self.conv(f, c[0]), c[1], act)
                z = self.dwconv(h, c[3])
                if s["se"]:
                    u = self.bn(z, c[4], ACT_NONE)
                    se = c[5]
                    y = self.gate(u, se.fc[0].weight, se.fc[0].bias, se.fc[2].weight, se.fc[2].bias, ACT_HSIGMOID, act, 0.0)
                else:
                    y = self.bn(z, c[4], act)
                f = self.bn(self.conv(y, c[7]), c[8], ACT_NONE, res=res)
            else:
                y = self.bn(self.dwconv(f, c[0]), c[1], act)
                if s["se"]:  # no-expand form: activation first, then SE (SURVEY F10)
                    se = c[3]
                    y = self.gate(y, se.fc[0].weight, se.fc[0].bias, se.fc[2].weight, se.fc[2].bias, ACT_HSIGMOID, ACT_NONE, 0.0)
                f = self.bn(self.conv(y, c[4]), c[5], ACT_NONE, res=res)
        return self.bn(self.conv(f, mob.conv[0]), mob.conv[1], ACT_HSWISH, out=out)

    def spatial_branch(self, x: torch.Tensor, xcol: Optional[Map], sb, out: Optional[Map] = None) -> Tuple[Map, Map]:
        """SpatialBranch ``sb`` (cabinet.py:108-129) on the fp32 NCHW ``x`` (``xcol``: its 7x7 im2col, or None for the
        CUDA-core stem) -> (sb.conv1's convolution output, the branch's output).  ``out``: where sb.conv_out's BN writes
        (CABiNet: channels [0:128] of the FFM concat buffer) or None."""
        stem7 = self.conv_stem(xcol, sb.conv1.conv) if xcol is not None else self.conv(None, sb.conv1.conv, nchw=x)
        s1 = self.bn(stem7, sb.conv1.bn, ACT_RELU)
        s2 = self.bn(self.conv(s1, sb.conv2.conv), sb.conv2.bn, ACT_RELU)
        s3 = self.bn(self.conv(s2, sb.conv3.conv), sb.conv3.bn, ACT_RELU)
        return stem7, self.bn(self.conv(s3, sb.conv_out.conv), sb.conv_out.bn, ACT_RELU, out=out)

    def attention_branch(self, cat: Map, x: Map, ab, low_path=None) -> Tuple[Map, Map]:
        """AttentionBranch ``ab`` (cabinet.py:75-94).  ``cat``: the b1 concat buffer [x | CAB feat] (cabinet.py:87); ``x``:
        its first channels, already written.  -> (low, high): convb's output and b4's fp32 class logits.  ``low_path(low)``
        runs right after convb (CABiNet: its x4 upsample into the FFM concat buffer)."""
        feat = self.bn(self.conv(x, ab.conva[0]), ab.conva[1], ACT_RELU)
        feat2 = cat.slice(x.C, feat.C)
        self.cab(feat, ab.a2block, feat2)
        low = self.conv(feat2, ab.convb)
        if low_path is not None:
            low_path(low)
        cat.needs_grad = x.needs_grad or feat2.needs_grad
        fused = self.bn(self.conv(cat, ab.b1), ab.b2, ACT_RELU)
        return low, self.conv(fused, ab.b4, out_dtype=torch.float32)

    def ffm(self, cat: Map, ffm) -> Map:
        """FeatureFusionModule ``ffm`` (cabinet.py:142-153) on ``cat`` = [fsp | fcp]: feat * atten + feat."""
        ff = self.bn(self.conv(cat, ffm.convblk.conv), ffm.convblk.bn, ACT_RELU)
        return self.gate(ff, ffm.conv1.weight, None, ffm.conv2.weight, None, ACT_SIGMOID, ACT_NONE, 1.0)

    def head(self, f: Map, head) -> Map:
        """CABiNetOutput ``head`` (cabinet.py:162-172) -> its fp32 class map."""
        hc = self.bn(self.conv(f, head.conv.conv), head.conv.bn, ACT_RELU)
        return self.conv(hc, head.conv_out, out_dtype=torch.float32)

    # ------------------------------------------------------------------ the step
    def forward(self, x: torch.Tensor, logits_dtype=torch.float32, input_grad: bool = False):
        """Train-mode ``CABiNet.forward`` (cabinet.py:207-247) -> (final_logit, high_res_logit_up), NCHW.  ``input_grad``:
        the backward also computes the gradient of ``x`` (``self.dx``)."""
        m = self.model
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()
        N, _, H, W = x.shape
        self.tape, self.launches, self.pgrads, self.phase = [], 0, {}, "fwd"
        self._pflat, self._bn_seen = None, []
        self._stems = (None, None, tuple(x.shape)) if input_grad else None
        mob, sb, ab, ffm, head = m.mobile, m.sb, m.ab, m.ffm, m.conv_out

        # ---- spatial branch (cabinet.py:108-129) -> channels [0:128] of the FFM concat buffer
        H8, W8 = _sb_hw(H, W)
        n_sb = sb.conv_out.conv.out_channels
        cat_ffm = self.new(N, H8, W8, n_sb + ab.convb.out_channels)
        xcol = self.stem_im2col(x) if (self.use_tc and self.stem_gemm) else None
        sb_lo = len(self.tape)
        stem7, sb_feat = self.spatial_branch(x, xcol, sb, out=cat_ffm.slice(0, n_sb))
        sb_hi = len(self.tape)

        # ---- backbone (mobilenetv3.py:102-159,202-205)
        stem3 = (self.conv_stem(xcol, mob.features[0][0]) if xcol is not None
                 else self.conv(None, mob.features[0][0], nchw=x))
        f = self.bn(stem3, mob.features[0][1], ACT_HSWISH)
        if input_grad:
            self._stems = (stem7, stem3, tuple(x.shape))
        h32, w32 = backbone_hw([blk.spec for blk in list(mob.features)[1:]], f.H, f.W)
        n_mf = mob.conv[0].out_channels
        cat_b1 = self.new(N, h32, w32, n_mf + 256)
        mf = self.mobilenet(f, mob, out=cat_b1.slice(0, n_mf))

        # ---- attention branch (cabinet.py:75-94, cab.py:131-162,175-184,213-216)
        def low_path(low):
            low_up = self.resample(low, "bilinear", H8, W8, out=cat_ffm.slice(n_sb, low.C))     # cabinet.py:228-233
            cat_ffm.needs_grad = sb_feat.needs_grad or low_up.needs_grad

        _, high = self.attention_branch(cat_b1, mf, ab, low_path)
        aux8 = self.resample(high, "bilinear", H8, W8)                                          # cabinet.py:234-239

        # ---- feature fusion + head (cabinet.py:142-153,162-172)
        # backward: once this convolution's data gradient exists, the spatial branch (tape[sb_lo:sb_hi]: big, bandwidth-
        # bound kernels) is independent of the attention branch / backbone (many small kernels): a branch of its own
        self._branch = (sb_lo, sb_hi, len(self.tape))
        final8 = self.head(self.ffm(cat_ffm, ffm), head)
        final, bwd_final = self.logits_up(final8, H, W, logits_dtype)
        aux, bwd_aux = self.logits_up(aux8, H, W, logits_dtype)
        self._out_bwd = (bwd_final, bwd_aux)
        if self._bn_seen:
            torch._foreach_add_(self._bn_seen, 1)
        return final, aux

    def backward(self, d_final: Optional[torch.Tensor], d_aux: Optional[torch.Tensor]) -> Dict[int, torch.Tensor]:
        """Gradients of the two logit tensors -> {id(parameter): fp32 gradient} for the parameters that require grad, and
        ``self.dx``: the fp32 NCHW gradient of the input when the forward was asked for it (else None)."""
        g = _Grads(self)
        self.pgrads, self.phase, self._pflat, self._side_used = {}, "bwd", None, False
        self._ensure_pflat()  # zero-filled on THIS stream before any branch adds into it
        for dy, bwd in ((d_final, self._out_bwd[0]), (d_aux, self._out_bwd[1])):
            if dy is not None:
                bwd(g, dy)
        on_gpu = torch.device(self.dev).type == "cuda"  # (the host-only dry run of the schedule has no streams)
        lo, hi, ready = self._branch if (self.branch_overlap and self.trace is None and self._branch and on_gpu) else (0, 0, -1)
        main = torch.cuda.current_stream(self.dev) if on_gpu else None
        for i in range(len(self.tape) - 1, -1, -1):
            if lo <= i < hi:
                continue  # ran on the branch stream
            self.tape[i](g)
            if i == ready:
                if self._side2 is None:
                    self._side2 = torch.cuda.Stream(self.dev)
                self._side2.wait_stream(main)
                with torch.cuda.stream(self._side2):
                    for j in range(hi - 1, lo - 1, -1):
                        self.tape[j](g)
        if hi > lo:
            main.wait_stream(self._side2)
        self.dx = self._stem_dgrad(g) if self._stems is not None else None
        if self._side_used:  # join: the parameter gradients are complete when the caller's stream continues
            main.wait_stream(self._side)
        self.tape = []
        return self.pgrads

    def _stem_dgrad(self, g: _Grads) -> Optional[torch.Tensor]:
        """dx of the network input: both stems' data gradients in one cabinet_stem_dgrad call, on the main stream once the
        spatial branch (sb.conv1's output gradient) has joined it.  None when neither stem received a gradient."""
        # stem7 None: a standalone MobileNetV3; stem3 None: a standalone SpatialBranch
        stem7, stem3, (N, _, H, W) = self._stems
        dy7 = g.get(stem7) if stem7 is not None else None
        dy3 = g.get(stem3) if stem3 is not None else None
        if dy7 is None and dy3 is None:
            return None
        dx = torch.empty((N, 3, H, W), dtype=torch.float32, device=self.dev)
        m = self.model
        w7 = getattr(m, "sb", m).conv1.conv.weight.data_ptr() if stem7 is not None else None
        w3 = getattr(m, "mobile", m).features[0][0].weight.data_ptr() if stem3 is not None else None
        dy = dy7 if dy7 is not None else dy3
        self._call("cabinet_stem_dgrad", dy7.ptr if dy7 is not None else None, dy7.ld if dy7 is not None else 0,
                   dy3.ptr if dy3 is not None else None, dy3.ld if dy3 is not None else 0, dy.dt, w7, w3, dx.data_ptr(),
                   N, H, W, dy.H, dy.W)
        return dx

    # ------------------------------------------------------------------ a standalone ContextAggregationBlock
    def _relayout(self, src: torch.Tensor, src_strides, dst: torch.Tensor, dst_strides, N, H, W, C):
        """dst = src between two (N, H, W, C) stride patterns and float dtypes (NCHW <-> NHWC at the block's boundary)."""
        if {src.dtype, dst.dtype} == {torch.bfloat16, torch.float16}:  # no kernel for this pair: through fp32
            tmp = torch.empty((N, H, W, C), dtype=torch.float32, device=self.dev)
            self._relayout(src, src_strides, tmp, (H * W * C, W * C, C, 1), N, H, W, C)
            src, src_strides = tmp, (H * W * C, W * C, C, 1)
        ty, tx = self.tables.get("identity", H, H, False), self.tables.get("identity", W, W, False)
        self._call("cabinet_resample_sep", src.data_ptr(), self._dt(src), *src_strides, dst.data_ptr(), self._dt(dst),
                   *dst_strides, N, H, W, C, *(t.data_ptr() for t in ty), *(t.data_ptr() for t in tx), 0)

    def block_forward(self, x: torch.Tensor, input_grad: bool) -> torch.Tensor:
        """``self.model`` is a ContextAggregationBlock: its train-mode (or differentiable eval-mode) forward on the
        (N, C, H, W) ``x`` -> y of x's shape and dtype; the tape is kept for ``block_backward``."""
        N, C, H, W = x.shape
        self.tape, self.launches, self.pgrads, self.phase = [], 0, {}, "fwd"
        self._pflat, self._bn_seen, self._stems = None, [], None
        nchw = lambda t: (t.stride(0), t.stride(2), t.stride(3), t.stride(1))  # noqa: E731  (n, y, x, c) strides
        feat, out = self.new(N, H, W, C), self.new(N, H, W, C)
        self._relayout(x, nchw(x), feat.t, (H * W * C, W * C, C, 1), N, H, W, C)
        feat.needs_grad = input_grad
        self.cab(feat, self.model, out)
        y = torch.empty_like(x, memory_format=torch.contiguous_format)
        self._relayout(out.t, (H * W * C, W * C, C, 1), y, nchw(y), N, H, W, C)
        self._block = (feat, out)
        if self._bn_seen:
            torch._foreach_add_(self._bn_seen, 1)
        return y

    def block_backward(self, dy: torch.Tensor) -> Tuple[Dict[int, torch.Tensor], Optional[torch.Tensor]]:
        """Gradient of ``block_forward``'s output -> ({id(parameter): fp32 gradient}, gradient of x in x's dtype or None)."""
        feat, out = self._block
        N, H, W, C = out.N, out.H, out.W, out.C
        g = _Grads(self)
        self.pgrads, self.phase, self._pflat, self._side_used = {}, "bwd", None, False
        self._ensure_pflat()
        dx = None
        if out.needs_grad:
            dout, _ = g.out(out)
            self._relayout(dy, (dy.stride(0), dy.stride(2), dy.stride(3), dy.stride(1)), dout.t, (H * W * C, W * C, C, 1),
                           N, H, W, C)
            for i in range(len(self.tape) - 1, -1, -1):
                self.tape[i](g)
            dfeat = g.get(feat) if feat.needs_grad else None
            if dfeat is not None:
                dx = torch.empty((N, C, H, W), dtype=dy.dtype, device=self.dev)
                self._relayout(dfeat.t, (H * W * C, W * C, C, 1), dx, (C * H * W, W, 1, H * W), N, H, W, C)
        if self._side_used:  # join: the parameter gradients are complete when the caller's stream continues
            torch.cuda.current_stream(self.dev).wait_stream(self._side)
        self.tape, self._block = [], None
        return self.pgrads, dx

    # ------------------------------------------------------------------ a standalone MobileNetV3
    def backbone_forward(self, x: torch.Tensor, input_grad: bool) -> torch.Tensor:
        """``self.model`` is a MobileNetV3: its train-mode (or differentiable eval-mode) forward on the (N, 3, H, W) ``x``
        -> (N, out_channels, h32, w32) NCHW in x's dtype; the tape is kept for ``backbone_backward``."""
        mob, xdt = self.model, x.dtype
        if x.dtype != torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()
        self.tape, self.launches, self.pgrads, self.phase = [], 0, {}, "fwd"
        self._pflat, self._bn_seen = None, []
        self._stems = (None, None, tuple(x.shape)) if input_grad else None
        stem = mob.features[0][0]
        k = stem.kernel_size[0]
        stem3 = (self.conv_stem(self.stem_im2col(x, k), stem, k) if self.use_tc and self.stem_gemm
                 else self.conv(None, stem, nchw=x))
        f = self.bn(stem3, mob.features[0][1], ACT_HSWISH)
        if input_grad:
            self._stems = (None, stem3, tuple(x.shape))
        out = self.mobilenet(f, mob)
        N, C, h, w = out.N, out.C, out.H, out.W
        y = torch.empty((N, C, h, w), dtype=xdt, device=self.dev)
        self._relayout(out.t, (h * w * C, w * C, C, 1), y, (C * h * w, w, 1, h * w), N, h, w, C)
        self._block = out
        if self._bn_seen:
            torch._foreach_add_(self._bn_seen, 1)
        return y

    def backbone_backward(self, dy: torch.Tensor) -> Tuple[Dict[int, torch.Tensor], Optional[torch.Tensor]]:
        """Gradient of ``backbone_forward``'s output -> ({id(parameter): fp32 gradient}, fp32 gradient of x or None)."""
        out = self._block
        N, H, W, C = out.N, out.H, out.W, out.C
        g = _Grads(self)
        self.pgrads, self.phase, self._pflat, self._side_used = {}, "bwd", None, False
        self._ensure_pflat()
        dx = None
        if out.needs_grad:
            dout, _ = g.out(out)
            self._relayout(dy, (dy.stride(0), dy.stride(2), dy.stride(3), dy.stride(1)), dout.t, (H * W * C, W * C, C, 1),
                           N, H, W, C)
            for i in range(len(self.tape) - 1, -1, -1):
                self.tape[i](g)
            dx = self._stem_dgrad(g) if self._stems is not None else None
        if self._side_used:  # join: the parameter gradients are complete when the caller's stream continues
            torch.cuda.current_stream(self.dev).wait_stream(self._side)
        self.tape, self._block, self._stems = [], None, None
        return self.pgrads, dx

    # ------------------------------------------------------------------ a standalone branch or head
    def _to_map(self, x: torch.Tensor, m: Map):
        """NCHW ``x`` -> the NHWC map ``m`` (a channel slice of a concat buffer, say), in m's dtype."""
        self._relayout(x, (x.stride(0), x.stride(2), x.stride(3), x.stride(1)), m.t[..., m.off:m.off + m.C],
                       (m.H * m.W * m.ld, m.W * m.ld, m.ld, 1), m.N, m.H, m.W, m.C)

    def _from_map(self, m: Map, dtype: torch.dtype) -> torch.Tensor:
        """The NHWC map ``m`` -> a new NCHW tensor of ``dtype``."""
        y = torch.empty((m.N, m.C, m.H, m.W), dtype=dtype, device=self.dev)
        self._relayout(m.t[..., m.off:m.off + m.C], (m.H * m.W * m.ld, m.W * m.ld, m.ld, 1), y,
                       (y.stride(0), y.stride(2), y.stride(3), y.stride(1)), m.N, m.H, m.W, m.C)
        return y

    def module_forward(self, xs, needs_grad) -> Tuple[List[torch.Tensor], tuple]:
        """``self.model`` is a standalone SpatialBranch, AttentionBranch, FeatureFusionModule or CABiNetOutput: its
        train-mode (or differentiable eval-mode) forward on the NCHW inputs ``xs`` -> its NCHW outputs in the first
        input's dtype, and the call's record (tape, boundary maps, stems) that ``module_backward`` takes.  The record belongs
        to the call, not the engine: several calls of one module before a backward (two inputs into one loss, activation
        checkpointing) each keep their own.  ``needs_grad[i]``: ``module_backward`` computes the gradient of ``xs[i]``.
        Inputs are written straight into the buffers the first layers read (the b1 / convblk concat buffers)."""
        from . import modules

        m, xdt = self.model, xs[0].dtype
        self.tape, self.launches, self.pgrads, self.phase = [], 0, {}, "fwd"
        self._pflat, self._bn_seen, self._stems = None, [], None
        N, _, H, W = xs[0].shape
        ins = []
        if isinstance(m, modules.SpatialBranch):
            x = xs[0] if xdt == torch.float32 and xs[0].is_contiguous() else xs[0].float().contiguous()
            self._stems = (None, None, tuple(x.shape)) if needs_grad[0] else None
            xcol = self.stem_im2col(x) if (self.use_tc and self.stem_gemm) else None
            stem7, out = self.spatial_branch(x, xcol, m)
            if needs_grad[0]:
                self._stems = (stem7, None, tuple(x.shape))
            outs = [out]
        elif isinstance(m, modules.AttentionBranch):
            cat = self.new(N, H, W, xs[0].shape[1] + m.conva[0].out_channels)
            x = cat.slice(0, xs[0].shape[1])
            self._to_map(xs[0], x)
            x.needs_grad = needs_grad[0]
            ins, outs = [x], list(self.attention_branch(cat, x, m))
        elif isinstance(m, modules.FeatureFusionModule):
            c1, c2 = xs[0].shape[1], xs[1].shape[1]
            cat = self.new(N, H, W, c1 + c2)
            ins = [cat.slice(0, c1), cat.slice(c1, c2)]
            for t, mp, rg in zip(xs, ins, needs_grad):
                self._to_map(t, mp)
                mp.needs_grad = rg
            cat.needs_grad = any(needs_grad)
            outs = [self.ffm(cat, m)]
        elif isinstance(m, modules.CABiNetOutput):
            f = self.new(N, H, W, xs[0].shape[1])
            self._to_map(xs[0], f)
            f.needs_grad = needs_grad[0]
            ins, outs = [f], [self.head(f, m)]
        else:
            raise TypeError(f"module_forward runs the branches and heads of CABiNet, not {type(m).__name__}")
        ys = [self._from_map(o, xdt) for o in outs]
        record = (self.tape, ins, outs, self._stems)
        self.tape, self._stems = [], None
        if self._bn_seen:
            torch._foreach_add_(self._bn_seen, 1)
        return ys, record

    def module_backward(self, record, dys, xdts) -> Tuple[Dict[int, torch.Tensor], List[Optional[torch.Tensor]]]:
        """Gradients of the outputs of the ``module_forward`` call that returned ``record`` (None: that output is unused,
        and layers only it reaches run no backward) -> ({id(parameter): fp32 gradient}, [gradient of each input in
        ``xdts[i]`` or None])."""
        self.tape, ins, outs, self._stems = record
        g = _Grads(self)
        self.pgrads, self.phase, self._pflat, self._side_used = {}, "bwd", None, False
        self._ensure_pflat()
        dxs = [None] * len(xdts)
        live = [(o, dy) for o, dy in zip(outs, dys) if dy is not None and o.needs_grad]
        if live:
            for o, dy in live:
                do, _ = g.out(o)
                self._to_map(dy, do)
            for i in range(len(self.tape) - 1, -1, -1):
                self.tape[i](g)
            if self._stems is not None:
                dx = self._stem_dgrad(g)
                dxs[0] = dx.to(xdts[0]) if dx is not None else None
            for i, mp in enumerate(ins):
                d = g.get(mp) if mp.needs_grad else None
                dxs[i] = self._from_map(d, xdts[i]) if d is not None else None
        if self._side_used:  # join: the parameter gradients are complete when the caller's stream continues
            torch.cuda.current_stream(self.dev).wait_stream(self._side)
        self.tape, self._stems = [], None
        return self.pgrads, dxs

    # ------------------------------------------------------------------ the step as two CUDA graphs
    def _addresses(self) -> tuple:
        """Everything a captured graph has baked in: parameter / buffer addresses, which parameters take a gradient and
        which BatchNorm modules use their batch statistics."""
        return (tuple((p.data_ptr(), p.requires_grad) for p in self.model.parameters()),
                tuple(b.data_ptr() for b in self.model.buffers()),
                tuple(m.training for m in self.model.modules() if isinstance(m, torch.nn.BatchNorm2d)))

    def step_forward(self, x: torch.Tensor, logits_dtype=torch.float32, input_grad: bool = False):
        """``forward`` for the autograd hand-off: eager for the first ``graph_after`` steps of a geometry, graph replay after."""
        self._active = None
        if not self.use_graph or self.trace is not None or torch.cuda.is_current_stream_capturing():
            return self.forward(x, logits_dtype, input_grad)
        key = (tuple(x.shape), logits_dtype, self.use_tc, self.wgrad_tc, self.stem_gemm, self.dgrad_s2_tc, self.attn_tc,
               self.wgrad_overlap, self.branch_overlap) + ((True,) if input_grad else ())
        addr = self._addresses()
        st = self._gsteps.get(key)
        if st is not None and st.fwd is not None and st.addr != addr:
            st = None  # parameters moved: the old graphs point at freed memory
        if st is None:
            st = self._gsteps[key] = _GraphedStep()
        if st.fwd is None:
            st.seen += 1
            if st.seen <= self.graph_after:
                return self.forward(x, logits_dtype, input_grad)
            captured = [k for k, v in self._gsteps.items() if v.fwd is not None]
            for k in captured[:max(0, len(captured) - self.max_graphs + 1)]:
                del self._gsteps[k]  # oldest geometries first: each one pins its activations in its own pool
            try:
                self._capture(st, x, logits_dtype, addr, input_grad)
            except Exception as e:  # e.g. out of memory for the pool: stay on the eager schedule, loudly
                import warnings

                warnings.warn(f"cabinet_b200: CUDA-graph capture of the training step failed ({e!r}); continuing eagerly")
                self.use_graph = False
                self._gsteps.clear()
                torch.cuda.synchronize(self.dev)
                return self.forward(x, logits_dtype, input_grad)
        st.x.copy_(x)
        st.fwd.replay()
        self.launches, self.phase = st.n_fwd, "fwd"
        self._active = st
        return st.final.detach(), st.aux.detach()  # fresh tensor objects: autograd attaches this step's node to them

    def step_backward(self, d_final: Optional[torch.Tensor],
                      d_aux: Optional[torch.Tensor]) -> Tuple[Dict[int, torch.Tensor], Optional[torch.Tensor]]:
        """-> (parameter gradients as ``backward`` returns them, the input gradient or None)."""
        st, self._active = self._active, None
        if st is None:
            return self.backward(d_final, d_aux), self.dx
        if d_final is None or d_aux is None:
            # an unused output: the eager backward over the captured forward's tape (its saved activations are the static
            # buffers the replay just filled) leaves the parameters only that output reaches without a gradient
            self.tape, self._out_bwd, self._branch, self._stems = list(st.tape), st.out_bwd, st.branch, st.stems
            return self.backward(d_final, d_aux), self.dx
        st.d_final.copy_(d_final)
        st.d_aux.copy_(d_aux)
        st.bwd.replay()
        self.launches += st.n_bwd
        # the next replay rewrites the static dx: hand autograd a copy, so a gradient the caller keeps stays as it is
        return st.grads, st.dx.clone() if st.dx is not None else None

    def _capture(self, st: "_GraphedStep", x: torch.Tensor, logits_dtype, addr: tuple, input_grad: bool):
        dev = self.dev
        st.x = torch.empty(tuple(x.shape), dtype=torch.float32, device=dev)
        st.x.copy_(x)
        fwd, bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        pool = torch.cuda.graph_pool_handle()
        # no cyclic garbage collection during the captures: a discarded model is a cycle (model <-> engine), and collecting
        # it destroys its CUDA graphs, which invalidates a capture in progress
        gc_enabled = gc.isenabled()
        gc.disable()
        try:
            with torch.cuda.graph(fwd, pool=pool, capture_error_mode="thread_local"):
                st.final, st.aux = self.forward(st.x, logits_dtype, input_grad)
            st.n_fwd = self.launches
            st.tape, st.out_bwd, st.branch = self.tape, self._out_bwd, self._branch  # keeps every saved activation alive
            st.stems = self._stems
            st.d_final, st.d_aux = torch.empty_like(st.final), torch.empty_like(st.aux)
            with torch.cuda.graph(bwd, pool=pool, capture_error_mode="thread_local"):
                st.grads = dict(self.backward(st.d_final, st.d_aux))
                st.dx = self.dx
        finally:
            if gc_enabled:
                gc.enable()
        st.n_bwd = self.launches - st.n_fwd
        st.fwd, st.bwd, st.addr = fwd, bwd, addr


class _GraphedStep:
    """Captured forward / backward graphs of one input geometry and their static buffers."""

    def __init__(self):
        self.seen = 0
        self.fwd = self.bwd = None
        self.x = self.final = self.aux = self.d_final = self.d_aux = None
        self.tape = self.out_bwd = self.grads = self.addr = self.branch = self.stems = self.dx = None
        self.n_fwd = self.n_bwd = 0


class TrainStep(torch.autograd.Function):
    """Autograd hand-off: inputs = (engine, logits dtype, x, *parameters); outputs = the two logit tensors.  The gradient
    of ``x`` is computed when ``x`` requires grad (autograd casts the fp32 result to ``x``'s dtype)."""

    @staticmethod
    def forward(ctx, eng: TrainEngine, logits_dtype, x, *params):
        with torch.no_grad(), torch.cuda.device(eng.dev):
            final, aux = eng.step_forward(x, logits_dtype, bool(ctx.needs_input_grad[2]))
        ctx.eng, ctx.params = eng, params
        return final, aux

    @staticmethod
    def backward(ctx, d_final, d_aux):
        eng = ctx.eng
        with torch.no_grad(), torch.cuda.device(eng.dev):
            grads, dx = eng.step_backward(d_final, d_aux)
        out = []
        for p in ctx.params:
            gp = grads.get(id(p))
            out.append(gp.to(p.dtype) if gp is not None else None)
        return (None, None, dx, *out)


class BlockStep(torch.autograd.Function):
    """Autograd hand-off of a standalone ContextAggregationBlock: inputs = (engine, x, *parameters); output = y."""

    @staticmethod
    def forward(ctx, eng: TrainEngine, x, *params):
        with torch.no_grad(), torch.cuda.device(eng.dev):
            y = eng.block_forward(x, bool(ctx.needs_input_grad[1]))
        ctx.eng, ctx.params = eng, params
        return y

    @staticmethod
    def backward(ctx, dy):
        eng = ctx.eng
        with torch.no_grad(), torch.cuda.device(eng.dev):
            grads, dx = eng.block_backward(dy)
        return (None, dx, *(grads[id(p)].to(p.dtype) if id(p) in grads else None for p in ctx.params))


class ModuleStep(torch.autograd.Function):
    """Autograd hand-off of a standalone module (``TrainEngine.module_forward``): inputs = (engine, k, k NCHW tensors,
    *parameters); outputs = the module's NCHW outputs in the first input's dtype.  An unused output's gradient stays None
    (no materialised zeros), and a gradient is returned for each input that requires one, in that input's dtype."""

    @staticmethod
    def forward(ctx, eng: TrainEngine, k: int, *args):
        xs, params = args[:k], args[k:]
        ctx.set_materialize_grads(False)
        with torch.no_grad(), torch.cuda.device(eng.dev):
            ys, ctx.record = eng.module_forward(xs, [bool(ctx.needs_input_grad[2 + i]) for i in range(k)])
        ctx.eng, ctx.params, ctx.xdts = eng, params, [x.dtype for x in xs]
        return tuple(ys)

    @staticmethod
    def backward(ctx, *dys):
        eng = ctx.eng
        if ctx.record is None:  # freed by the first backward, as PyTorch frees a node's saved tensors
            raise RuntimeError("Trying to backward through a cabinet_b200 module's graph a second time: its saved "
                               "activations were freed by the first backward")
        with torch.no_grad(), torch.cuda.device(eng.dev):
            grads, dxs = eng.module_backward(ctx.record, dys, ctx.xdts)
        ctx.record = None
        return (None, None, *dxs, *(grads[id(p)].to(p.dtype) if id(p) in grads else None for p in ctx.params))


class BackboneStep(torch.autograd.Function):
    """Autograd hand-off of a standalone MobileNetV3: inputs = (engine, x, *parameters); output = the feature map.  The
    gradient of ``x`` is computed when ``x`` requires grad and returned in x's dtype."""

    @staticmethod
    def forward(ctx, eng: TrainEngine, x, *params):
        with torch.no_grad(), torch.cuda.device(eng.dev):
            y = eng.backbone_forward(x, bool(ctx.needs_input_grad[1]))
        ctx.eng, ctx.params, ctx.xdt = eng, params, x.dtype
        return y

    @staticmethod
    def backward(ctx, dy):
        eng = ctx.eng
        with torch.no_grad(), torch.cuda.device(eng.dev):
            grads, dx = eng.backbone_backward(dy)
        dx = dx.to(ctx.xdt) if dx is not None else None
        return (None, dx, *(grads[id(p)].to(p.dtype) if id(p) in grads else None for p in ctx.params))

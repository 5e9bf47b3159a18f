"""GPU: every variant of the training step's tensor-core convolutions, weight packers, layout helpers, attention softmax,
CUDA-core forward kernels and eval-mode BatchNorm statistics that the step launches, replayed against float64
references.

One case per variant key of ``tests/train_variants.py`` (the plan the host dispatch derives: flat or tiled walk, TW x TH
patch and output tails, ragged K blocks, N / M tiles, resident weights, finalize kernel, channel chunks, windows,
residual aliasing), with the smallest geometry the step records for that key (``tests/test_train_variants_cpu.py``
checks that the matrix covers every key).  Operands, canaries and the launch come from ``tests/test_gpu_train_variants``:

* every strided operand is a channel window of a NaN-filled buffer at the recorded pixel stride and alignment, so a map
  that reads a channel past ``C`` (channels 5..7 of the ``Cin = 5, ldx = 8`` classifier gradient) turns the output into
  NaN; bytes outside the output windows must stay bit-unchanged and inputs must not change at all;
* the scratch of ``conv_wgrad_tc`` is exactly ``cabinet_conv_wgrad_tc_scratch_floats`` long, followed by a canary block;
* in-place cases pass the same buffer as ``res`` and ``y``, as the step does; accumulating outputs (``conv_wgrad_tc``
  ``dw``, ``embed_filter`` extract-add) start from random priors; biases and ``alpha`` are random, not the step's zeros;
* the tensor-core GEMMs read the weights that ``cabinet_pack_conv_weight`` packs into a NaN-prefilled buffer (a pad
  element left unwritten poisons the output), and the reference uses those packed, rounded weights;
* the call runs twice and must give bit-identical outputs.

Bounds:

* GEMM-like outputs (convolutions, ``gate_fc``, the attention GEMMs): elementwise
  ``|got - ref| <= 2^-16 * mag + u(ref)`` with ``mag`` the same operation on ``|x|``, ``|w|`` (plus ``|bias|``,
  ``|res|``) in float64, ``u`` one ulp of a 2-byte output type (0 for fp32 outputs), plus ``2^-23 * |prior|`` when the
  output accumulates and 2 ulp of fp32 after a non-linear gate activation evaluated in fp32.  A single wrong tap, border
  pixel or 64-channel K block exceeds it by orders of magnitude;
* data movement (packs, ``im2col_nchw``, ``transpose_tokens``, ``embed_filter``, ``pack_dw_weight``): bit-exact against
  torch's round-to-nearest conversion, padding ``+0.0``;
* ``attn_softmax``: ``p_half`` is bit-exactly ``p`` rounded to the operand type; ``p``, ``softmax_rows``,
  ``cab_combine``, ``upsample_logits_nchw`` and ``bn_frozen_stats`` follow ``tests/test_gpu_train_variants.py``: fp32
  rel-L2 < 1e-5, 2-byte outputs within 2 ulp plus ``1e-6 * max|ref|``; ``attn_softmax_backward`` the same as
  ``softmax_backward``.
"""

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from cabinet_b200 import _lib  # noqa: E402
from cabinet_b200._lib import F32  # noqa: E402
from tests.test_gpu_train_variants import ITD, LEAD, TD, Case, Operand, _launch, act_ref, compare, nchw, rows_of, stream, ulp  # noqa: E402
from tests.train_variants import variant_key  # noqa: E402

EPS_MAG = 2.0 ** -16


def _c(a, b):
    return -(-a // b) * b


def gemm_expect(k, name, op, ref, mag, extra=0.0):
    """op (+ its prior) within 2^-16 * mag + 1 ulp of its type (+ 2^-23 |prior|) of the float64 reference."""
    ref = ref.reshape(op.rows, op.C)
    bound = EPS_MAG * mag.reshape(op.rows, op.C) + extra
    if op.prior is not None:
        bound = bound + 2.0 ** -23 * op.prior.abs()
        ref = ref + op.prior
    if op.dt != torch.float32:
        bound = bound + ulp(ref.to(op.dt).double(), op.dt)
    k.checks.append((name, op, ref, bound))


def exact_expect(k, name, op, ref):
    """op must be bit-identical to the float64 ``ref`` rounded (to nearest) to the operand type."""
    k.checks.append((name, op, ref.reshape(op.rows, op.C), "exact"))


def check(name, op, ref, how):
    if isinstance(how, torch.Tensor):
        got = op.got()
        assert torch.isfinite(got).all(), f"{name}: {int((~torch.isfinite(got)).sum())} non-finite values"
        err = (got - ref).abs()
        bad = (err > how).nonzero()
        if bad.numel():
            i = tuple(bad[0].tolist())
            ratio = float((err / how).max())
            raise AssertionError(f"{name}: {bad.shape[0]} of {got.numel()} elements beyond the bound (worst {ratio:.3g}x), "
                                 f"first {list(i)}: got {float(got[i])}, reference {float(ref[i])}, bound {float(how[i]):.3g}")
    elif how == "exact":
        want = ref.to(op.dt).cpu().view(ITD[op.dt])
        got = op.view.detach().reshape(op.rows, op.C).cpu().view(ITD[op.dt])
        bad = (got != want).nonzero()
        assert bad.numel() == 0, f"{name}: {bad.shape[0]} of {got.numel()} elements not bit-exact, first {bad[0].tolist()}: " \
                                 f"got {float(op.got()[tuple(bad[0])])}, want {float(ref[tuple(bad[0])])}"
    elif callable(how):
        how()
    else:
        compare(name, op, ref, how)


def _cuda(t):
    return t.cuda()


def conv_ref(x4, w4, stride, pad, bias=None, groups=1):
    """float64 convolution (on the GPU) of the rounded operands and the same of their magnitudes -> ([N][C][H][W]) x 2."""
    x4, w4 = _cuda(x4), _cuda(w4)
    ref = F.conv2d(x4, w4, None, stride, pad, groups=groups)
    mag = F.conv2d(x4.abs(), w4.abs(), None, stride, pad, groups=groups)
    if bias is not None:
        b = _cuda(bias).reshape(1, -1, 1, 1)
        ref, mag = ref + b, mag + b.abs()
    return ref.cpu(), mag.cpu()


def packed_weights(lib, k, Cout, Cin, KH, KW, dt):
    """cabinet_pack_conv_weight of random OIHW weights into a NaN-prefilled [ceil16(Cout)][taps][ceil64(Cin)] buffer of
    type dt -> (device buffer, the packed weights as float64 OIHW [Cout][Cin][KH][KW])."""
    r16, k64, taps = _c(Cout, 16), _c(Cin, 64), KH * KW
    w = k.rnd(Cout, Cin, KH, KW, scale=(Cin * taps) ** -0.5).float().cuda()
    wp = torch.full((r16 * taps * k64,), float("nan"), dtype=TD[dt], device="cuda")
    _lib.check(lib.cabinet_pack_conv_weight(w.data_ptr(), Cout, Cin, KH, KW, wp.data_ptr(), dt, r16, k64, 0, stream()),
               "pack_conv_weight")
    torch.cuda.synchronize()
    k.keep.append((w, wp))
    packed = wp.double().cpu().reshape(r16, taps, k64)
    return wp, packed[:Cout, :, :Cin].reshape(Cout, KH, KW, Cin).permute(0, 3, 1, 2)


class StridedOut(Operand):
    """An output written through a strided pixel view of a larger NHWC buffer: pixel (n, oh, ow) at pixel
    first + n * sn + oh * sh + ow * sw; every other byte of the buffer is a canary."""

    def __init__(self, total_px, first, N, OH, OW, sw, sh, sn, C, ld, dtype):
        super().__init__(total_px, C, ld, 0, dtype, None, out=True)
        base = LEAD + first * ld
        self.view = self.buf[base:].as_strided((N, OH, OW, C), (sn * ld, sh * ld, sw * ld, 1))
        self.mask.zero_()
        self.mask[base:].as_strided((N, OH, OW, C), (sn * ld, sh * ld, sw * ld, 1)).fill_(True)
        self.rows, self.ptr = N * OH * OW, self.view.data_ptr()

    def got(self):
        return self.view.double().cpu().reshape(self.rows, self.C)


# ----------------------------------------------------------------------------------------------------------- runners
def _tc_common(lib, a, k, Cin, Cout, op):
    N, H, W = a["N"], a["H"], a["W"]
    x = k.inp(N * H * W, Cin, a["ldx"], a["x"], op, k.rnd(N * H * W, Cin))
    bias = k.vec(k.rnd(Cout, scale=0.5))
    return N, H, W, x, bias


def run_conv_tc(lib, a, k):
    Cin, Cout, KH, KW, s, pad, op = (a[n] for n in ("Cin", "Cout", "KH", "KW", "stride", "pad", "op_dtype"))
    N, H, W, x, bias = _tc_common(lib, a, k, Cin, Cout, op)
    OH, OW, ydt = a["OH"], a["OW"], a["y_dtype"]
    assert a["act"] == 0
    wp, w4 = packed_weights(lib, k, Cout, Cin, KH, KW, op)
    ref, mag = conv_ref(nchw(x.ref, N, H, W), w4, s, pad, bias.ref[0])
    ref, mag = rows_of(ref), rows_of(mag)
    res = None
    if a["res_is_y"]:   # the stride-1 data gradient accumulating into dx in place: res = y
        assert a["ldres"] == a["ldy"] and ydt == op
        y = k.out(N * OH * OW, Cout, a["ldy"], a["y"], ydt, acc=True)
        res = y
        gemm_expect(k, "y", y, ref, mag + y.prior.abs())
    else:
        if a["res"] is not None:
            res = k.inp(N * OH * OW, Cout, a["ldres"], a["res"], op, k.rnd(N * OH * OW, Cout))
            ref, mag = ref + res.ref, mag + res.ref.abs()
        y = k.out(N * OH * OW, Cout, a["ldy"], a["y"], ydt)
        gemm_expect(k, "y", y, ref, mag)
    return lambda: lib.cabinet_conv_tc_dt(x.ptr, a["ldx"], N, H, W, Cin, wp.data_ptr(), Cout, KH, KW, s, pad, bias.ptr,
                                          None if res is None else res.ptr, a["ldres"], y.ptr, ydt, a["ldy"], OH, OW, 0, op,
                                          stream())


def run_conv_tc_view(lib, a, k):
    Cin, Cout, KH, KW, pad, op = (a[n] for n in ("Cin", "Cout", "KH", "KW", "pad", "op_dtype"))
    N, H, W, x, bias = _tc_common(lib, a, k, Cin, Cout, op)
    OH, OW, sw, sh, sn = a["OH"], a["OW"], a["y_sw"], a["y_sh"], a["y_sn"]
    assert sw == 2
    Wd = sh // 2
    Hd = sn // Wd
    # the odd parity class where it fits (a view that starts one row / pixel into dx), else the even one
    py, px = int(2 * OH <= Hd), int(2 * OW <= Wd)
    wp, w4 = packed_weights(lib, k, Cout, Cin, KH, KW, op)
    # the last rows / columns of an odd parity class read past the end of dy: zeros, as on the leading side
    eh, ew = max(pad, OH + KH - 1 - H - pad), max(pad, OW + KW - 1 - W - pad)
    ref, mag = conv_ref(F.pad(nchw(x.ref, N, H, W), (pad, ew, pad, eh)), w4, 1, 0, bias.ref[0])
    ref, mag = rows_of(ref[:, :, :OH, :OW]), rows_of(mag[:, :, :OH, :OW])
    y = StridedOut(N * sn, py * Wd + px, N, OH, OW, sw, sh, sn, Cout, a["ldy"], op)
    k.ops.append(y)
    gemm_expect(k, "y", y, ref, mag)
    return lambda: lib.cabinet_conv_tc_view_dt(x.ptr, a["ldx"], N, H, W, Cin, wp.data_ptr(), Cout, KH, KW, pad, bias.ptr,
                                               y.ptr, a["ldy"], OH, OW, sw, sh, sn, op, stream())


def run_conv_tc_imgw(lib, a, k):
    Cin, Cout, op, ydt = a["Cin"], a["Cout"], a["op_dtype"], a["y_dtype"]
    N, H, W, x, bias = _tc_common(lib, a, k, Cin, Cout, op)
    assert (a["KH"], a["KW"], a["stride"], a["pad"], a["res"]) == (1, 1, 1, 0, None) and a["w_image_stride"] == Cout * Cin
    w = k.inp(N * Cout, Cin, Cin, a["w_packed_per_image"], op, k.rnd(N * Cout, Cin, scale=Cin ** -0.5))
    xs, ws = x.ref.reshape(N, H * W, Cin), w.ref.reshape(N, Cout, Cin)
    ref = torch.einsum("npc,noc->npo", xs, ws) + bias.ref[0]
    mag = torch.einsum("npc,noc->npo", xs.abs(), ws.abs()) + bias.ref[0].abs()
    y = k.out(N * H * W, Cout, a["ldy"], a["y"], ydt)
    gemm_expect(k, "y", y, ref, mag)
    return lambda: lib.cabinet_conv_tc_imgw_dt(x.ptr, a["ldx"], N, H, W, Cin, w.ptr, a["w_image_stride"], Cout, 1, 1, 1, 0,
                                               bias.ptr, None, 0, y.ptr, ydt, a["ldy"], H, W, 0, op, stream())


def wgrad_scratch(k, n):
    """The documented scratch size exactly, with the canary block of an Operand behind it."""
    sc = Operand(1, n, n, 0, F32, None, out=True)
    k.ops.append(sc)
    return sc


def run_conv_wgrad_tc(lib, a, k):
    N, H, W, Cin, Cout, KH, KW, s, pad, op = (a[n] for n in ("N", "H", "W", "Cin", "Cout", "KH", "KW", "stride", "pad",
                                                             "op_dtype"))
    OH, OW = (H + 2 * pad - KH) // s + 1, (W + 2 * pad - KW) // s + 1
    dy = k.inp(N * OH * OW, Cout, a["lddy"], a["dy"], op, k.rnd(N * OH * OW, Cout))
    x = k.inp(N * H * W, Cin, a["ldx"], a["x"], op, k.rnd(N * H * W, Cin))
    dw = k.out(Cout, Cin * KH * KW, Cin * KH * KW, 0, F32, acc=True)
    x4, dy4 = _cuda(nchw(x.ref, N, H, W)), _cuda(nchw(dy.ref, N, OH, OW))
    ref = torch.nn.grad.conv2d_weight(x4, (Cout, Cin, KH, KW), dy4, s, pad).cpu()
    mag = torch.nn.grad.conv2d_weight(x4.abs(), (Cout, Cin, KH, KW), dy4.abs(), s, pad).cpu()
    gemm_expect(k, "dw", dw, ref, mag)
    sc = wgrad_scratch(k, int(lib.cabinet_conv_wgrad_tc_scratch_floats(N, H, W, Cin, Cout, KH, KW, s, pad)))
    return lambda: lib.cabinet_conv_wgrad_tc_dt(dy.ptr, a["lddy"], x.ptr, a["ldx"], dw.ptr, N, H, W, Cin, Cout, KH, KW, s, pad,
                                                sc.ptr, op, stream())


def run_conv_wgrad_tc_batched(lib, a, k):
    N, H, W, Cin, Cout, op = (a[n] for n in ("N", "H", "W", "Cin", "Cout", "op_dtype"))
    P = H * W
    A = k.inp(N * P, Cout, a["lda"], a["a"], op, k.rnd(N * P, Cout))
    x = k.inp(N * P, Cin, a["ldx"], a["x"], op, k.rnd(N * P, Cin))
    out = k.out(N * Cout, Cin, Cin, 0, F32)
    As, xs = A.ref.reshape(N, P, Cout), x.ref.reshape(N, P, Cin)
    gemm_expect(k, "out", out, torch.einsum("npo,npc->noc", As, xs), torch.einsum("npo,npc->noc", As.abs(), xs.abs()))
    return lambda: lib.cabinet_conv_wgrad_tc_batched_dt(A.ptr, a["lda"], x.ptr, a["ldx"], out.ptr, N, H, W, Cin, Cout, op,
                                                        stream())


def _dw_common(a, k, dt):
    N, H, W, C, kk, s, OH, OW = (a[n] for n in ("N", "H", "W", "C", "k", "stride", "OH", "OW"))
    assert a["act"] == 0 and a["gap_sum"] is None
    x = k.inp(N * H * W, C, a["ldx"], a["x"], dt, k.rnd(N * H * W, C))
    w = k.vec(k.rnd(kk * kk, C, scale=1.0 / kk))
    bias = k.vec(k.rnd(C, scale=0.5))
    w4 = w.ref.reshape(kk * kk, C).t().reshape(C, 1, kk, kk)
    ref, mag = conv_ref(nchw(x.ref, N, H, W), w4, s, (kk - 1) // 2, bias.ref[0], groups=C)
    y = k.out(N * OH * OW, C, a["ldy"], a["y"], dt)
    gemm_expect(k, "y", y, rows_of(ref), rows_of(mag))
    return N, H, W, C, kk, s, OH, OW, x, w, bias, y


def run_dwconv_tma(lib, a, k):
    N, H, W, C, kk, s, OH, OW, x, w, bias, y = _dw_common(a, k, a["op_dtype"])
    return lambda: lib.cabinet_dwconv_tma_dt(x.ptr, a["ldx"], w.ptr, bias.ptr, y.ptr, a["ldy"], N, H, W, C, kk, s, OH, OW, 0,
                                             None, a["op_dtype"], stream())


def run_dwconv(lib, a, k):
    N, H, W, C, kk, s, OH, OW, x, w, bias, y = _dw_common(a, k, a["dtype"])
    return lambda: lib.cabinet_dwconv(x.ptr, a["ldx"], w.ptr, bias.ptr, y.ptr, a["ldy"], a["dtype"], N, H, W, C, kk, s, OH, OW,
                                      0, None, stream())


def run_pack_conv_weight(lib, a, k):
    Cout, Cin, KH, KW, rp, kp, flip, dt = (a[n] for n in ("Cout", "Cin", "KH", "KW", "rows_pad", "k_pad", "transpose_flip",
                                                         "out_dtype"))
    taps = KH * KW
    w = k.vec(k.rnd(Cout * Cin * taps))
    w4 = w.ref.reshape(Cout, Cin, taps)
    want = torch.zeros(rp, taps, kp, dtype=torch.float64)
    if flip:   # rows = input channels, taps mirrored, k = output channels
        want[:Cin, :, :Cout] = w4.flip(2).permute(1, 2, 0)
    else:
        want[:Cout, :, :Cin] = w4.permute(0, 2, 1)
    out = k.out(1, want.numel(), want.numel(), a["out"], dt)
    exact_expect(k, "out", out, want)
    return lambda: lib.cabinet_pack_conv_weight(w.ptr, Cout, Cin, KH, KW, out.ptr, dt, rp, kp, flip, stream())


def run_pack_conv_weight_parity(lib, a, k):
    Cout, Cin, K, pad, py, px, KH2, KW2, pad2, rp, kp, dt = (a[n] for n in (
        "Cout", "Cin", "K", "pad", "py", "px", "KH2", "KW2", "pad2", "rows_pad", "k_pad", "out_dtype"))
    w = k.vec(k.rnd(Cout * Cin * K * K))
    w4 = w.ref.reshape(Cout, Cin, K, K)
    want = torch.zeros(rp, KH2, KW2, kp, dtype=torch.float64)
    for jy in range(KH2):
        for jx in range(KW2):
            ky, kx = py + pad - 2 * (jy - pad2), px + pad - 2 * (jx - pad2)
            if 0 <= ky < K and 0 <= kx < K:
                want[:Cin, jy, jx, :Cout] = w4[:, :, ky, kx].t()
    out = k.out(1, want.numel(), want.numel(), a["out"], dt)
    exact_expect(k, "out", out, want)
    return lambda: lib.cabinet_pack_conv_weight_parity_dt(w.ptr, Cout, Cin, K, pad, py, px, KH2, KW2, pad2, out.ptr, rp, kp,
                                                          dt, stream())


def run_pack_dw_weight(lib, a, k):
    C, kk, flip = a["C"], a["k"], a["flip"]
    w = k.vec(k.rnd(C * kk * kk))
    want = w.ref.reshape(C, kk * kk).t()
    out = k.out(kk * kk, C, C, a["out"], F32)
    exact_expect(k, "out", out, want.flip(0) if flip else want)
    return lambda: lib.cabinet_pack_dw_weight(w.ptr, C, kk, flip, out.ptr, stream())


def run_embed_filter(lib, a, k):
    Cout, Cin, kk, K, ld = a["Cout"], a["Cin"], a["k"], a["K"], a["ld_big"]
    o = (K - kk) // 2
    if a["extract_add"]:   # w_small += the embedded taps of w_big
        big = k.inp(Cout, ld, ld, a["w_big"], F32, k.rnd(Cout, ld))
        small = k.out(1, Cout * Cin * kk * kk, Cout * Cin * kk * kk, a["w_small"], F32, acc=True)
        taps = big.ref[:, :Cin * K * K].reshape(Cout, Cin, K, K)[:, :, o:o + kk, o:o + kk].reshape(1, -1)
        want = (small.prior.float() + taps.float()).double()   # one fp32 addition, round to nearest
        exact_expect(k, "w_small", small, want)
        return lambda: lib.cabinet_embed_filter(small.ptr, Cout, Cin, kk, K, big.ptr, ld, 1, stream())
    small = k.inp(1, Cout * Cin * kk * kk, Cout * Cin * kk * kk, a["w_small"], F32, k.rnd(1, Cout * Cin * kk * kk))
    big = k.out(Cout, ld, ld, a["w_big"], F32, acc=True)   # the taps are overwritten, everything else keeps its prior
    taps = big.prior[:, :Cin * K * K].reshape(Cout, Cin, K, K).clone()
    taps[:, :, o:o + kk, o:o + kk] = small.ref.reshape(Cout, Cin, kk, kk)
    want = big.prior.clone()
    want[:, :Cin * K * K] = taps.reshape(Cout, -1)
    exact_expect(k, "w_big", big, want)
    return lambda: lib.cabinet_embed_filter(small.ptr, Cout, Cin, kk, K, big.ptr, ld, 0, stream())


def run_im2col_nchw(lib, a, k):
    N, Cin, H, W, kk, s, pad, ld, dt = (a[n] for n in ("N", "Cin", "H", "W", "k", "stride", "pad", "ld", "out_dtype"))
    OH, OW = (H + 2 * pad - kk) // s + 1, (W + 2 * pad - kk) // s + 1
    x = k.inp(1, N * Cin * H * W, N * Cin * H * W, a["x"], F32, k.rnd(1, N * Cin * H * W))
    cols = F.unfold(x.ref.reshape(N, Cin, H, W), kk, padding=pad, stride=s)   # [N][Cin*k*k][OH*OW], OIHW column order
    want = torch.zeros(N * OH * OW, ld, dtype=torch.float64)
    want[:, :Cin * kk * kk] = cols.permute(0, 2, 1).reshape(N * OH * OW, -1)
    out = k.out(N * OH * OW, ld, ld, a["out"], dt)
    exact_expect(k, "out", out, want)
    return lambda: lib.cabinet_im2col_nchw_dt(x.ptr, N, Cin, H, W, kk, s, pad, out.ptr, ld, dt, stream())


def run_transpose_tokens(lib, a, k):
    N, L, C, dt = a["N"], a["L"], a["C"], a["op_dtype"]
    x = k.inp(N * L, C, a["ldx"], a["x"], dt, k.rnd(N * L, C))
    out = k.out(N * C, L, L, a["out"], dt)
    exact_expect(k, "out", out, x.ref.reshape(N, L, C).transpose(1, 2).reshape(N * C, L))
    return lambda: lib.cabinet_transpose_tokens_dt(x.ptr, a["ldx"], out.ptr, N, L, C, dt, stream())


def run_attn_softmax(lib, a, k):
    rows, cols, dt = a["rows"], a["cols"], a["op_dtype"]
    scale = a["scale"] * 1.3
    s = k.inp(rows, cols, cols, a["s"], F32, k.rnd(rows, cols, scale=8.0))
    p = k.out(rows, cols, cols, a["p"], F32)
    ph = k.out(rows, cols, cols, a["p_half"], dt)
    k.checks.append(("p", p, torch.softmax(s.ref * float(torch.tensor(scale, dtype=torch.float32)), -1), 1e-5))

    def p_half_is_p_rounded():
        want = p.view.detach().to(ph.dt).view(ITD[ph.dt])
        assert torch.equal(ph.view.detach().view(ITD[ph.dt]), want), "p_half is not p rounded to the operand type"

    k.checks.append(("p_half", ph, None, p_half_is_p_rounded))
    return lambda: lib.cabinet_attn_softmax_dt(s.ptr, scale, p.ptr, ph.ptr, rows, cols, dt, stream())


def run_attn_softmax_backward(lib, a, k):
    rows, cols, dt = a["rows"], a["cols"], a["op_dtype"]
    alpha = a["alpha"] * 1.3
    p = k.inp(rows, cols, cols, a["p"], F32, torch.softmax(k.rnd(rows, cols, scale=3.0), -1))
    dp = k.inp(rows, cols, cols, a["dp"], F32, k.rnd(rows, cols))
    ds = k.out(rows, cols, cols, a["ds_half"], dt)
    al = float(torch.tensor(alpha, dtype=torch.float32))
    k.checks.append(("ds", ds, p.ref * (dp.ref - (dp.ref * p.ref).sum(-1, keepdim=True)) * al, 1e-5))
    return lambda: lib.cabinet_attn_softmax_backward_dt(p.ptr, dp.ptr, ds.ptr, rows, cols, alpha, dt, stream())


def _flat_operand(k, extent, al, dtype):
    return k.inp(1, extent, extent, al, dtype, k.rnd(1, extent))


def run_conv2d_simt(lib, a, k):
    B, N, H, W, Cin, Cout, KH, KW, s, pad, OH, OW = (a[n] for n in (
        "batches", "N", "H", "W", "Cin", "Cout", "KH", "KW", "stride", "pad", "OH", "OW"))
    assert a["res"] is None and a["act"] == 0
    sxn, sxh, sxw, sxc, xbs = a["sxn"], a["sxh"], a["sxw"], a["sxc"], a["x_batch_stride"]
    alpha = 1.0 if a["alpha"] == 1 else a["alpha"] * 1.3
    al32 = float(torch.tensor(alpha, dtype=torch.float32))
    if sxc == 1 and sxh == W * sxw and sxn == H * sxh and xbs in (0, N * sxn):   # NHWC rows (a channel window)
        x = k.inp(B * N * H * W, Cin, sxw, a["x"], a["x_dtype"], k.rnd(B * N * H * W, Cin))
        X = x.ref.reshape(B, N, H, W, Cin)
    else:   # any other layout: a dense buffer, gathered with the strides
        ext = (B - 1) * xbs + (N - 1) * sxn + (H - 1) * sxh + (W - 1) * sxw + (Cin - 1) * sxc + 1
        x = _flat_operand(k, ext, a["x"], a["x_dtype"])
        X = torch.stack([x.ref[0, b * xbs:].as_strided((N, H, W, Cin), (sxn, sxh, sxw, sxc)) for b in range(B)])
    K, sco, sk, wbs = KH * KW * Cin, a["w_sco"], a["w_sk"], a["w_batch_stride"]
    w = _flat_operand(k, (B - 1) * wbs + (Cout - 1) * sco + (K - 1) * sk + 1, a["w"], a["w_dtype"])
    Wt = torch.stack([w.ref[0, b * wbs:].as_strided((Cout, K), (sco, sk)) for b in range(B)])
    Wt = Wt.reshape(B, Cout, KH, KW, Cin).permute(0, 1, 4, 2, 3)
    bias = k.vec(k.rnd(Cout, scale=0.5)) if a["bias"] is not None else None
    M = N * OH * OW
    assert B == 1 or a["y_batch_stride"] == M * a["ldy"]   # the batches' outputs are consecutive rows
    refs, mags = [], []
    for b in range(B):
        r, m = conv_ref(X[b].permute(0, 3, 1, 2), Wt[b], s, pad)
        refs.append(rows_of(r) * al32)
        mags.append(rows_of(m) * abs(al32))
    ref, mag = torch.cat(refs), torch.cat(mags)
    if bias is not None:
        ref, mag = ref + bias.ref[0], mag + bias.ref[0].abs()
    y = k.out(B * M, Cout, a["ldy"], a["y"], a["y_dtype"])
    gemm_expect(k, "y", y, ref, mag)
    return lambda: lib.cabinet_conv2d_simt(x.ptr, a["x_dtype"], sxn, sxh, sxw, sxc, xbs, w.ptr, a["w_dtype"], sco, sk, wbs,
                                           None if bias is None else bias.ptr, None, 0, y.ptr, a["y_dtype"], a["ldy"],
                                           a["y_batch_stride"], B, N, H, W, Cin, Cout, KH, KW, s, pad, OH, OW, 0, alpha, stream())


def run_gate_fc(lib, a, k):
    N, C, J, act = a["N"], a["C"], a["J"], a["act"]
    assert not a["in_fixed"]
    sc = a["in_scale"]
    x = k.inp(N, C, C, a["in"], F32, k.rnd(N, C, scale=1.0 / sc))
    Wm = k.inp(J, C, C, a["W"], F32, k.rnd(J, C, scale=C ** -0.5))
    b = k.vec(k.rnd(J, scale=0.5)) if a["b"] is not None else None
    xs = x.ref * float(torch.tensor(sc, dtype=torch.float32))
    pre = xs @ Wm.ref.t() + (0 if b is None else b.ref[0])
    mag = xs.abs() @ Wm.ref.abs().t() + (0 if b is None else b.ref[0].abs())
    ref = act_ref(pre, act)
    out = k.out(N, J, J, a["out"], F32)
    gemm_expect(k, "out", out, ref, mag, extra=2.0 ** -22 * ref.abs())   # the gate evaluated in fp32
    return lambda: lib.cabinet_gate_fc(x.ptr, sc, Wm.ptr, None if b is None else b.ptr, out.ptr, N, C, J, act, 0, stream())


def run_cab_combine(lib, a, k):
    n, C, dt = a["n_pixels"], a["C"], a["dtype"]
    g, x, r = (k.inp(n, C, C, 0, dt, k.rnd(n, C, scale=2.0)) for _ in range(3))
    gamma = k.vec(torch.tensor([0.7]))
    out = k.out(n, C, a["ldo"], a["out"], dt)
    k.checks.append(("out", out, gamma.ref[0, 0] * g.ref + x.ref + x.ref * torch.sigmoid(r.ref), 1e-5))
    return lambda: lib.cabinet_cab_combine(g.ptr, x.ptr, r.ptr, out.ptr, a["ldo"], gamma.ptr, dt, n, C, stream())


def run_softmax_rows(lib, a, k):
    rows, cols, dt = a["rows"], a["cols"], a["p_dtype"]
    s = k.inp(rows, cols, cols, a["s"], F32, k.rnd(rows, cols, scale=3.0))
    p = k.out(rows, cols, cols, a["p"], dt)
    k.checks.append(("p", p, torch.softmax(s.ref, -1), 1e-5))
    return lambda: lib.cabinet_softmax_rows(s.ptr, p.ptr, dt, rows, cols, stream())


def run_upsample_logits_nchw(lib, a, k):
    N, IH, IW, C, OH, OW, dt = (a[n] for n in ("N", "IH", "IW", "C", "OH", "OW", "y_dtype"))
    x = k.inp(N * IH * IW, C, C, a["x"], F32, k.rnd(N * IH * IW, C))
    y = k.out(N * C * OH, OW, OW, a["y"], dt)
    ref = F.interpolate(nchw(x.ref, N, IH, IW), size=(OH, OW), mode="bilinear", align_corners=False)
    k.checks.append(("y", y, ref.reshape(N * C * OH, OW), 1e-5))
    return lambda: lib.cabinet_upsample_logits_nchw(x.ptr, N, IH, IW, C, y.ptr, dt, OH, OW, stream())


def run_bn_frozen_stats(lib, a, k):
    C, eps = a["C"], a["eps"]
    gamma = k.vec(k.rnd(C, scale=0.3, shift=1.0)) if a["gamma"] is not None else None
    beta = k.vec(k.rnd(C, scale=0.2)) if a["beta"] is not None else None
    rm, rv = k.vec(k.rnd(C)), k.vec(k.rnd(C).abs() + 0.1)
    stats = k.out(4, C, C, 0, F32)
    g = gamma.ref[0] if gamma is not None else 1.0
    bt = beta.ref[0] if beta is not None else 0.0
    invstd = (rv.ref[0] + float(torch.tensor(eps, dtype=torch.float32))).rsqrt()
    k.checks.append(("stats", stats, torch.stack([rm.ref[0], invstd, g * invstd, bt - rm.ref[0] * g * invstd]), 1e-6))
    p = lambda o: None if o is None else o.ptr  # noqa: E731
    return lambda: lib.cabinet_bn_frozen_stats(p(gamma), p(beta), rm.ptr, rv.ptr, eps, C, stats.ptr, stream())


RUNNERS = {name[4:]: fn for name, fn in globals().items() if name.startswith("run_")}

# One case per variant key: the smallest recorded call of each (tests/test_train_variants_cpu.py lists any key
# the step reaches that is missing here, with an example call).
CASES = [
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 32, 'W': 64, 'Cin': 128, 'w_packed': 0, 'Cout': 64, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 64, 'OH': 32,
                 'OW': 64, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 128, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 128, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 256, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 640, 'N': 2, 'H': 8, 'W': 16, 'Cin': 640, 'w_packed': 0, 'Cout': 128, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 128, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 1216, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 1216, 'y': 0, 'y_dtype': 1, 'ldy': 1216, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 152, 'N': 2, 'H': 32, 'W': 48, 'Cin': 152, 'w_packed': 0, 'Cout': 64, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 64, 'OH': 32,
                 'OW': 48, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 72, 'N': 2, 'H': 16, 'W': 24, 'Cin': 72, 'w_packed': 0, 'Cout': 16, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 16, 'OH': 16,
                 'OW': 24, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 120, 'N': 2, 'H': 32, 'W': 64, 'Cin': 120, 'w_packed': 0, 'Cout': 40, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 40, 'y': 0, 'y_dtype': 1, 'ldy': 40, 'OH': 32,
                 'OW': 64, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 80, 'N': 2, 'H': 16, 'W': 32, 'Cin': 80, 'w_packed': 0, 'Cout': 184, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 184, 'OH': 16,
                 'OW': 32, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 184, 'N': 2, 'H': 16, 'W': 32, 'Cin': 184, 'w_packed': 0, 'Cout': 80, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 80, 'y': 0, 'y_dtype': 1, 'ldy': 80, 'OH': 16,
                 'OW': 32, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 672, 'N': 2, 'H': 8, 'W': 16, 'Cin': 672, 'w_packed': 0, 'Cout': 160, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 160, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 672, 'N': 2, 'H': 16, 'W': 32, 'Cin': 672, 'w_packed': 0, 'Cout': 112, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 112, 'y': 0, 'y_dtype': 1, 'ldy': 112, 'OH': 16,
                 'OW': 32, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 160, 'N': 2, 'H': 8, 'W': 16, 'Cin': 160, 'w_packed': 0, 'Cout': 960, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 960, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 160, 'N': 2, 'H': 8, 'W': 16, 'Cin': 160, 'w_packed': 0, 'Cout': 672, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 672, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 24, 'N': 2, 'H': 64, 'W': 128, 'Cin': 24, 'w_packed': 0, 'Cout': 64, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 64, 'OH': 64,
                 'OW': 128, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 8, 'N': 2, 'H': 8, 'W': 16, 'Cin': 5, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 16, 'N': 2, 'H': 16, 'W': 24, 'Cin': 16, 'w_packed': 0, 'Cout': 16, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 16, 'OH': 16,
                 'OW': 24, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 16, 'N': 2, 'H': 16, 'W': 24, 'Cin': 16, 'w_packed': 0, 'Cout': 72, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 72, 'OH': 16,
                 'OW': 24, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 24, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 24, 'OH': 64,
                 'OW': 128, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 960, 'N': 2, 'H': 8, 'W': 16, 'Cin': 960, 'w_packed': 0, 'Cout': 160, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 160, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 960, 'N': 2, 'H': 8, 'W': 16, 'Cin': 960, 'w_packed': 0, 'Cout': 160, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 160, 'y': 0, 'y_dtype': 1, 'ldy': 160, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128, 'w_packed': 0, 'Cout': 640, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 640, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 8, 'W': 12, 'Cin': 128, 'w_packed': 0, 'Cout': 64, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 64, 'OH': 8,
                 'OW': 12, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 128, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 128, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 2, 'W': 3, 'Cin': 128, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 256, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 640, 'N': 2, 'H': 2, 'W': 3, 'Cin': 640, 'w_packed': 0, 'Cout': 128, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 128, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 832, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 832, 'y': 0, 'y_dtype': 1, 'ldy': 832, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 96, 'N': 2, 'H': 4, 'W': 6, 'Cin': 96, 'w_packed': 0, 'Cout': 40, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 40, 'OH': 4,
                 'OW': 6, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 144, 'N': 2, 'H': 4, 'W': 6, 'Cin': 144, 'w_packed': 0, 'Cout': 48, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 48, 'y': 0, 'y_dtype': 1, 'ldy': 48, 'OH': 4,
                 'OW': 6, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 288, 'N': 2, 'H': 2, 'W': 3, 'Cin': 288, 'w_packed': 0, 'Cout': 96, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 96, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 96, 'N': 2, 'H': 2, 'W': 3, 'Cin': 96, 'w_packed': 0, 'Cout': 576, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 576, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 96, 'N': 2, 'H': 2, 'W': 3, 'Cin': 96, 'w_packed': 0, 'Cout': 288, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 288, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 8, 'N': 2, 'H': 2, 'W': 3, 'Cin': 8, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 40, 'N': 2, 'H': 4, 'W': 6, 'Cin': 40, 'w_packed': 0, 'Cout': 96, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 96, 'OH': 4,
                 'OW': 6, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 48, 'N': 2, 'H': 4, 'W': 6, 'Cin': 48, 'w_packed': 0, 'Cout': 288, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 288, 'OH': 4,
                 'OW': 6, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 576, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576, 'w_packed': 0, 'Cout': 96, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 96, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 576, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576, 'w_packed': 0, 'Cout': 96, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 96, 'y': 0, 'y_dtype': 1, 'ldy': 96, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 2, 'W': 3, 'Cin': 128, 'w_packed': 0, 'Cout': 640, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 640, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 1216, 'N': 2, 'H': 8, 'W': 16, 'Cin': 1216, 'w_packed': 0, 'Cout': 256, 'KH': 3,
                 'KW': 3, 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 256,
                 'OH': 8, 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 1216, 'N': 2, 'H': 8, 'W': 16, 'Cin': 960, 'w_packed': 0, 'Cout': 256, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 1216, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 1216, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 960, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': 0, 'ldres': 1216, 'y': 0, 'y_dtype': 1, 'ldy': 1216, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 12, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 8,
                 'OW': 12, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 32, 'W': 64, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 32,
                 'OW': 64, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 832, 'N': 2, 'H': 2, 'W': 3, 'Cin': 832, 'w_packed': 0, 'Cout': 256, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 832, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576, 'w_packed': 0, 'Cout': 256, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 256, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 832, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 832, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 576, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': 0, 'ldres': 832, 'y': 0, 'y_dtype': 1, 'ldy': 832, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 64, 'N': 2, 'H': 128, 'W': 256, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 3, 'KW': 3,
                 'stride': 2, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 64, 'OH': 64,
                 'OW': 128, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 3, 'KW': 3,
                 'stride': 2, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 64, 'OH': 8,
                 'OW': 12, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 3, 'KW': 3,
                 'stride': 2, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 64, 'OH': 32,
                 'OW': 64, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 64, 'N': 2, 'H': 32, 'W': 48, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 3, 'KW': 3,
                 'stride': 2, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 64, 'OH': 16,
                 'OW': 24, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 5, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 5, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 8, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 8, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 32, 'W': 64, 'Cin': 128, 'w_packed': 0, 'Cout': 64, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 64, 'OH': 32,
                 'OW': 64, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 128, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 128, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 256, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 640, 'N': 2, 'H': 8, 'W': 16, 'Cin': 640, 'w_packed': 0, 'Cout': 128, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 128, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 1216, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 1216, 'y': 0, 'y_dtype': 2, 'ldy': 1216, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 152, 'N': 2, 'H': 32, 'W': 48, 'Cin': 152, 'w_packed': 0, 'Cout': 64, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 64, 'OH': 32,
                 'OW': 48, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 72, 'N': 2, 'H': 16, 'W': 24, 'Cin': 72, 'w_packed': 0, 'Cout': 16, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 16, 'OH': 16,
                 'OW': 24, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 120, 'N': 2, 'H': 32, 'W': 64, 'Cin': 120, 'w_packed': 0, 'Cout': 40, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 40, 'y': 0, 'y_dtype': 2, 'ldy': 40, 'OH': 32,
                 'OW': 64, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 80, 'N': 2, 'H': 16, 'W': 32, 'Cin': 80, 'w_packed': 0, 'Cout': 184, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 184, 'OH': 16,
                 'OW': 32, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 184, 'N': 2, 'H': 16, 'W': 32, 'Cin': 184, 'w_packed': 0, 'Cout': 80, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 80, 'y': 0, 'y_dtype': 2, 'ldy': 80, 'OH': 16,
                 'OW': 32, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 672, 'N': 2, 'H': 8, 'W': 16, 'Cin': 672, 'w_packed': 0, 'Cout': 160, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 160, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 672, 'N': 2, 'H': 16, 'W': 32, 'Cin': 672, 'w_packed': 0, 'Cout': 112, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 112, 'y': 0, 'y_dtype': 2, 'ldy': 112, 'OH': 16,
                 'OW': 32, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 160, 'N': 2, 'H': 8, 'W': 16, 'Cin': 160, 'w_packed': 0, 'Cout': 960, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 960, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 160, 'N': 2, 'H': 8, 'W': 16, 'Cin': 160, 'w_packed': 0, 'Cout': 672, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 672, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 24, 'N': 2, 'H': 64, 'W': 128, 'Cin': 24, 'w_packed': 0, 'Cout': 64, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 64, 'OH': 64,
                 'OW': 128, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 8, 'N': 2, 'H': 8, 'W': 16, 'Cin': 5, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 16, 'N': 2, 'H': 16, 'W': 24, 'Cin': 16, 'w_packed': 0, 'Cout': 16, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 16, 'OH': 16,
                 'OW': 24, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 16, 'N': 2, 'H': 16, 'W': 24, 'Cin': 16, 'w_packed': 0, 'Cout': 72, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 72, 'OH': 16,
                 'OW': 24, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 24, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 24, 'OH': 64,
                 'OW': 128, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 960, 'N': 2, 'H': 8, 'W': 16, 'Cin': 960, 'w_packed': 0, 'Cout': 160, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 160, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 960, 'N': 2, 'H': 8, 'W': 16, 'Cin': 960, 'w_packed': 0, 'Cout': 160, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 160, 'y': 0, 'y_dtype': 2, 'ldy': 160, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128, 'w_packed': 0, 'Cout': 640, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 640, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 8, 'W': 12, 'Cin': 128, 'w_packed': 0, 'Cout': 64, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 64, 'OH': 8,
                 'OW': 12, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 128, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 128, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 2, 'W': 3, 'Cin': 128, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 256, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 640, 'N': 2, 'H': 2, 'W': 3, 'Cin': 640, 'w_packed': 0, 'Cout': 128, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 128, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 832, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 832, 'y': 0, 'y_dtype': 2, 'ldy': 832, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 96, 'N': 2, 'H': 4, 'W': 6, 'Cin': 96, 'w_packed': 0, 'Cout': 40, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 40, 'OH': 4,
                 'OW': 6, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 144, 'N': 2, 'H': 4, 'W': 6, 'Cin': 144, 'w_packed': 0, 'Cout': 48, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 48, 'y': 0, 'y_dtype': 2, 'ldy': 48, 'OH': 4,
                 'OW': 6, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 288, 'N': 2, 'H': 2, 'W': 3, 'Cin': 288, 'w_packed': 0, 'Cout': 96, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 96, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 96, 'N': 2, 'H': 2, 'W': 3, 'Cin': 96, 'w_packed': 0, 'Cout': 576, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 576, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 96, 'N': 2, 'H': 2, 'W': 3, 'Cin': 96, 'w_packed': 0, 'Cout': 288, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 288, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 8, 'N': 2, 'H': 2, 'W': 3, 'Cin': 8, 'w_packed': 0, 'Cout': 256, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 40, 'N': 2, 'H': 4, 'W': 6, 'Cin': 40, 'w_packed': 0, 'Cout': 96, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 96, 'OH': 4,
                 'OW': 6, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 48, 'N': 2, 'H': 4, 'W': 6, 'Cin': 48, 'w_packed': 0, 'Cout': 288, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 288, 'OH': 4,
                 'OW': 6, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 576, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576, 'w_packed': 0, 'Cout': 96, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 96, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 576, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576, 'w_packed': 0, 'Cout': 96, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': 0, 'ldres': 96, 'y': 0, 'y_dtype': 2, 'ldy': 96, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 128, 'N': 2, 'H': 2, 'W': 3, 'Cin': 128, 'w_packed': 0, 'Cout': 640, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 640, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 1216, 'N': 2, 'H': 8, 'W': 16, 'Cin': 1216, 'w_packed': 0, 'Cout': 256, 'KH': 3,
                 'KW': 3, 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 256,
                 'OH': 8, 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 1216, 'N': 2, 'H': 8, 'W': 16, 'Cin': 960, 'w_packed': 0, 'Cout': 256, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 1216, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 1216, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 960, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': 0, 'ldres': 1216, 'y': 0, 'y_dtype': 2, 'ldy': 1216, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 12, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 8,
                 'OW': 12, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 32, 'W': 64, 'Cin': 256, 'w_packed': 0, 'Cout': 256, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 32,
                 'OW': 64, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 832, 'N': 2, 'H': 2, 'W': 3, 'Cin': 832, 'w_packed': 0, 'Cout': 256, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 832, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576, 'w_packed': 0, 'Cout': 256, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 256, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 832, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 832, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 576, 'KH': 3, 'KW': 3,
                 'stride': 1, 'pad': 1, 'bias': 0, 'res': 0, 'ldres': 832, 'y': 0, 'y_dtype': 2, 'ldy': 832, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': True}),
    ('conv_tc', {'x': 0, 'ldx': 64, 'N': 2, 'H': 128, 'W': 256, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 3, 'KW': 3,
                 'stride': 2, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 64, 'OH': 64,
                 'OW': 128, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 3, 'KW': 3,
                 'stride': 2, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 64, 'OH': 8,
                 'OW': 12, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 3, 'KW': 3,
                 'stride': 2, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 64, 'OH': 32,
                 'OW': 64, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 64, 'N': 2, 'H': 32, 'W': 48, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 3, 'KW': 3,
                 'stride': 2, 'pad': 1, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 64, 'OH': 16,
                 'OW': 24, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256, 'w_packed': 0, 'Cout': 5, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 5, 'OH': 8,
                 'OW': 16, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc', {'x': 0, 'ldx': 256, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256, 'w_packed': 0, 'Cout': 8, 'KH': 1, 'KW': 1,
                 'stride': 1, 'pad': 0, 'bias': 0, 'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 8, 'OH': 2,
                 'OW': 3, 'act': 0, 'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 64, 'OW': 128, 'y_sw': 2, 'y_sh': 512,
                      'y_sn': 32768, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 8, 'W': 12, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 8, 'OW': 12, 'y_sw': 2, 'y_sh': 48,
                      'y_sn': 384, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 32, 'W': 64, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 32, 'OW': 64, 'y_sw': 2, 'y_sh': 256,
                      'y_sn': 8192, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 16, 'OW': 24, 'y_sw': 2, 'y_sh': 96,
                      'y_sn': 1536, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 64, 'OW': 128, 'y_sw': 2, 'y_sh': 512,
                      'y_sn': 32768, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 8, 'W': 12, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 8, 'OW': 12, 'y_sw': 2, 'y_sh': 48,
                      'y_sn': 384, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 32, 'W': 64, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 32, 'OW': 64, 'y_sw': 2, 'y_sh': 256,
                      'y_sn': 8192, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 16, 'OW': 24, 'y_sw': 2, 'y_sh': 96,
                      'y_sn': 1536, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 64, 'OW': 128, 'y_sw': 2, 'y_sh': 512,
                      'y_sn': 32768, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 8, 'W': 12, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 8, 'OW': 12, 'y_sw': 2, 'y_sh': 48,
                      'y_sn': 384, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 32, 'W': 64, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 32, 'OW': 64, 'y_sw': 2, 'y_sh': 256,
                      'y_sn': 8192, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 16, 'OW': 24, 'y_sw': 2, 'y_sh': 96,
                      'y_sn': 1536, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 64, 'OW': 128, 'y_sw': 2, 'y_sh': 512,
                      'y_sn': 32768, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 8, 'W': 12, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 8, 'OW': 12, 'y_sw': 2, 'y_sh': 48,
                      'y_sn': 384, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 32, 'W': 64, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 32, 'OW': 64, 'y_sw': 2, 'y_sh': 256,
                      'y_sn': 8192, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 16, 'OW': 24, 'y_sw': 2, 'y_sh': 96,
                      'y_sn': 1536, 'op_dtype': 1}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 64, 'OW': 128, 'y_sw': 2, 'y_sh': 512,
                      'y_sn': 32768, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 8, 'W': 12, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 8, 'OW': 12, 'y_sw': 2, 'y_sh': 48,
                      'y_sn': 384, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 32, 'W': 64, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 32, 'OW': 64, 'y_sw': 2, 'y_sh': 256,
                      'y_sn': 8192, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 16, 'OW': 24, 'y_sw': 2, 'y_sh': 96,
                      'y_sn': 1536, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 64, 'OW': 128, 'y_sw': 2, 'y_sh': 512,
                      'y_sn': 32768, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 8, 'W': 12, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 8, 'OW': 12, 'y_sw': 2, 'y_sh': 48,
                      'y_sn': 384, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 32, 'W': 64, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 32, 'OW': 64, 'y_sw': 2, 'y_sh': 256,
                      'y_sn': 8192, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 1,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 16, 'OW': 24, 'y_sw': 2, 'y_sh': 96,
                      'y_sn': 1536, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 64, 'OW': 128, 'y_sw': 2, 'y_sh': 512,
                      'y_sn': 32768, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 8, 'W': 12, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 8, 'OW': 12, 'y_sw': 2, 'y_sh': 48,
                      'y_sn': 384, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 32, 'W': 64, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 32, 'OW': 64, 'y_sw': 2, 'y_sh': 256,
                      'y_sn': 8192, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 1, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 16, 'OW': 24, 'y_sw': 2, 'y_sh': 96,
                      'y_sn': 1536, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 64, 'OW': 128, 'y_sw': 2, 'y_sh': 512,
                      'y_sn': 32768, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 8, 'W': 12, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 8, 'OW': 12, 'y_sw': 2, 'y_sh': 48,
                      'y_sn': 384, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 32, 'W': 64, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 32, 'OW': 64, 'y_sw': 2, 'y_sh': 256,
                      'y_sn': 8192, 'op_dtype': 2}),
    ('conv_tc_view', {'x': 0, 'ldx': 64, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64, 'w_packed': 0, 'Cout': 64, 'KH': 2,
                      'KW': 2, 'pad': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'OH': 16, 'OW': 24, 'y_sw': 2, 'y_sh': 96,
                      'y_sn': 1536, 'op_dtype': 2}),
    ('conv_tc_imgw', {'x': 0, 'ldx': 128, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128, 'w_packed_per_image': 0,
                      'w_image_stride': 16384, 'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'bias': 0,
                      'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 128, 'OH': 8, 'OW': 16, 'act': 0,
                      'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc_imgw', {'x': 0, 'ldx': 128, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128, 'w_packed_per_image': 0,
                      'w_image_stride': 16384, 'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'bias': 0,
                      'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 128, 'OH': 8, 'OW': 16, 'act': 0,
                      'op_dtype': 1, 'res_is_y': False}),
    ('conv_tc_imgw', {'x': 0, 'ldx': 128, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128, 'w_packed_per_image': 0,
                      'w_image_stride': 16384, 'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'bias': 0,
                      'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 128, 'OH': 8, 'OW': 16, 'act': 0,
                      'op_dtype': 2, 'res_is_y': False}),
    ('conv_tc_imgw', {'x': 0, 'ldx': 128, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128, 'w_packed_per_image': 0,
                      'w_image_stride': 16384, 'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'bias': 0,
                      'res': None, 'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 128, 'OH': 8, 'OW': 16, 'act': 0,
                      'op_dtype': 2, 'res_is_y': False}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 40, 'x': 0, 'ldx': 72, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 64, 'Cin': 72,
                       'Cout': 40, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 184, 'x': 0, 'ldx': 80, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 32, 'Cin': 80,
                       'Cout': 184, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 16, 'x': 0, 'ldx': 152, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 48, 'Cin': 152,
                       'Cout': 16, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 112, 'x': 0, 'ldx': 480, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 32, 'Cin': 480,
                       'Cout': 112, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 64, 'Cin': 64,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 16, 'x': 0, 'ldx': 16, 'dw_oihw': 0, 'N': 2, 'H': 128, 'W': 256, 'Cin': 16,
                       'Cout': 16, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 24, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64,
                       'Cout': 24, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 240, 'x': 0, 'ldx': 40, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 64, 'Cin': 40,
                       'Cout': 240, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 24, 'x': 0, 'ldx': 72, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 12, 'Cin': 72,
                       'Cout': 24, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 128, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128,
                       'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 672, 'x': 0, 'ldx': 112, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 32, 'Cin': 112,
                       'Cout': 672, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 256, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 960, 'x': 0, 'ldx': 160, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 160,
                       'Cout': 960, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 1216, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256,
                       'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 640, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 640,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 112, 'x': 0, 'ldx': 672, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 32, 'Cin': 672,
                       'Cout': 112, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 384, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 12, 'Cin': 384,
                       'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 160, 'x': 0, 'ldx': 672, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 672,
                       'Cout': 160, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 160, 'x': 0, 'ldx': 960, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 960,
                       'Cout': 160, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 12, 'Cin': 64,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 16, 'x': 0, 'ldx': 16, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 24, 'Cin': 16,
                       'Cout': 16, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 40, 'x': 0, 'ldx': 96, 'dw_oihw': 0, 'N': 2, 'H': 4, 'W': 6, 'Cin': 96,
                       'Cout': 40, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 128, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 128,
                       'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 576, 'x': 0, 'ldx': 96, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 96,
                       'Cout': 576, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 256, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 48, 'x': 0, 'ldx': 144, 'dw_oihw': 0, 'N': 2, 'H': 4, 'W': 6, 'Cin': 144,
                       'Cout': 48, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 832, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256,
                       'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 640, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 640,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 96, 'x': 0, 'ldx': 288, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 288,
                       'Cout': 96, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 96, 'x': 0, 'ldx': 576, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576,
                       'Cout': 96, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 120, 'x': 0, 'ldx': 40, 'dw_oihw': 0, 'N': 2, 'H': 4, 'W': 6, 'Cin': 40,
                       'Cout': 120, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 144, 'x': 0, 'ldx': 48, 'dw_oihw': 0, 'N': 2, 'H': 4, 'W': 6, 'Cin': 48,
                       'Cout': 144, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 1216, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 1216,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 1216, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 960,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 256, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 12, 'Cin': 256,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 832, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 832,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 832, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 256, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 64, 'Cin': 256,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 64, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64,
                       'Cout': 64, 'KH': 3, 'KW': 3, 'stride': 2, 'pad': 1, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 64, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64,
                       'Cout': 64, 'KH': 3, 'KW': 3, 'stride': 2, 'pad': 1, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 64, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 48, 'Cin': 64,
                       'Cout': 64, 'KH': 3, 'KW': 3, 'stride': 2, 'pad': 1, 'op_dtype': 1}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 40, 'x': 0, 'ldx': 72, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 64, 'Cin': 72,
                       'Cout': 40, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 184, 'x': 0, 'ldx': 80, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 32, 'Cin': 80,
                       'Cout': 184, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 16, 'x': 0, 'ldx': 152, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 48, 'Cin': 152,
                       'Cout': 16, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 112, 'x': 0, 'ldx': 480, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 32, 'Cin': 480,
                       'Cout': 112, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 64, 'Cin': 64,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 16, 'x': 0, 'ldx': 16, 'dw_oihw': 0, 'N': 2, 'H': 128, 'W': 256, 'Cin': 16,
                       'Cout': 16, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 24, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64,
                       'Cout': 24, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 240, 'x': 0, 'ldx': 40, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 64, 'Cin': 40,
                       'Cout': 240, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 24, 'x': 0, 'ldx': 72, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 12, 'Cin': 72,
                       'Cout': 24, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 128, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128,
                       'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 672, 'x': 0, 'ldx': 112, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 32, 'Cin': 112,
                       'Cout': 672, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 256, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 960, 'x': 0, 'ldx': 160, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 160,
                       'Cout': 960, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 1216, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 256,
                       'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 640, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 640,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 112, 'x': 0, 'ldx': 672, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 32, 'Cin': 672,
                       'Cout': 112, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 384, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 12, 'Cin': 384,
                       'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 160, 'x': 0, 'ldx': 672, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 672,
                       'Cout': 160, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 160, 'x': 0, 'ldx': 960, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 960,
                       'Cout': 160, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 12, 'Cin': 64,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 16, 'x': 0, 'ldx': 16, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 24, 'Cin': 16,
                       'Cout': 16, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 40, 'x': 0, 'ldx': 96, 'dw_oihw': 0, 'N': 2, 'H': 4, 'W': 6, 'Cin': 96,
                       'Cout': 40, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 128, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 128,
                       'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 576, 'x': 0, 'ldx': 96, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 96,
                       'Cout': 576, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 256, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 48, 'x': 0, 'ldx': 144, 'dw_oihw': 0, 'N': 2, 'H': 4, 'W': 6, 'Cin': 144,
                       'Cout': 48, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 832, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 256,
                       'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 128, 'x': 0, 'ldx': 640, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 640,
                       'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 96, 'x': 0, 'ldx': 288, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 288,
                       'Cout': 96, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 96, 'x': 0, 'ldx': 576, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576,
                       'Cout': 96, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 120, 'x': 0, 'ldx': 40, 'dw_oihw': 0, 'N': 2, 'H': 4, 'W': 6, 'Cin': 40,
                       'Cout': 120, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 144, 'x': 0, 'ldx': 48, 'dw_oihw': 0, 'N': 2, 'H': 4, 'W': 6, 'Cin': 48,
                       'Cout': 144, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 1216, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 1216,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 1216, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 960,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 256, 'dw_oihw': 0, 'N': 2, 'H': 8, 'W': 12, 'Cin': 256,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 832, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 832,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 832, 'dw_oihw': 0, 'N': 2, 'H': 2, 'W': 3, 'Cin': 576,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 256, 'x': 0, 'ldx': 256, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 64, 'Cin': 256,
                       'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 64, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 16, 'W': 24, 'Cin': 64,
                       'Cout': 64, 'KH': 3, 'KW': 3, 'stride': 2, 'pad': 1, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 64, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 64, 'W': 128, 'Cin': 64,
                       'Cout': 64, 'KH': 3, 'KW': 3, 'stride': 2, 'pad': 1, 'op_dtype': 2}),
    ('conv_wgrad_tc', {'dy': 0, 'lddy': 64, 'x': 0, 'ldx': 64, 'dw_oihw': 0, 'N': 2, 'H': 32, 'W': 48, 'Cin': 64,
                       'Cout': 64, 'KH': 3, 'KW': 3, 'stride': 2, 'pad': 1, 'op_dtype': 2}),
    ('conv_wgrad_tc_batched', {'a': 0, 'lda': 128, 'x': 0, 'ldx': 128, 'out': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128,
                               'Cout': 128, 'op_dtype': 1}),
    ('conv_wgrad_tc_batched', {'a': 0, 'lda': 128, 'x': 0, 'ldx': 128, 'out': 0, 'N': 2, 'H': 8, 'W': 16, 'Cin': 128,
                               'Cout': 128, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 16, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 16, 'N': 2, 'H': 128, 'W': 256, 'C': 16,
                    'k': 3, 'stride': 1, 'OH': 128, 'OW': 256, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 72, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 72, 'N': 2, 'H': 64, 'W': 128, 'C': 72, 'k': 3,
                    'stride': 1, 'OH': 64, 'OW': 128, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 200, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 200, 'N': 2, 'H': 16, 'W': 32, 'C': 200,
                    'k': 3, 'stride': 1, 'OH': 16, 'OW': 32, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 480, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 480, 'N': 2, 'H': 16, 'W': 32, 'C': 480,
                    'k': 3, 'stride': 1, 'OH': 16, 'OW': 32, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 88, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 88, 'N': 2, 'H': 8, 'W': 12, 'C': 88, 'k': 3,
                    'stride': 1, 'OH': 8, 'OW': 12, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 184, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 184, 'N': 2, 'H': 16, 'W': 32, 'C': 184,
                    'k': 3, 'stride': 1, 'OH': 16, 'OW': 32, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 256, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 256, 'N': 2, 'H': 8, 'W': 16, 'C': 256,
                    'k': 3, 'stride': 1, 'OH': 8, 'OW': 16, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 256, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 256, 'N': 2, 'H': 2, 'W': 3, 'C': 256, 'k': 3,
                    'stride': 1, 'OH': 2, 'OW': 3, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 16, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 16, 'N': 2, 'H': 32, 'W': 48, 'C': 16, 'k': 3,
                    'stride': 2, 'OH': 16, 'OW': 24, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 72, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 72, 'N': 2, 'H': 16, 'W': 24, 'C': 72, 'k': 3,
                    'stride': 2, 'OH': 8, 'OW': 12, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 240, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 240, 'N': 2, 'H': 32, 'W': 64, 'C': 240,
                    'k': 3, 'stride': 2, 'OH': 16, 'OW': 32, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 64, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'N': 2, 'H': 128, 'W': 256, 'C': 64,
                    'k': 3, 'stride': 2, 'OH': 64, 'OW': 128, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 144, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 144, 'N': 2, 'H': 4, 'W': 6, 'C': 144, 'k': 5,
                    'stride': 1, 'OH': 4, 'OW': 6, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 240, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 240, 'N': 2, 'H': 4, 'W': 6, 'C': 240, 'k': 5,
                    'stride': 1, 'OH': 4, 'OW': 6, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 120, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 120, 'N': 2, 'H': 32, 'W': 64, 'C': 120,
                    'k': 5, 'stride': 1, 'OH': 32, 'OW': 64, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 120, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 120, 'N': 2, 'H': 4, 'W': 6, 'C': 120, 'k': 5,
                    'stride': 1, 'OH': 4, 'OW': 6, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 960, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 960, 'N': 2, 'H': 8, 'W': 16, 'C': 960,
                    'k': 5, 'stride': 1, 'OH': 8, 'OW': 16, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 576, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 576, 'N': 2, 'H': 2, 'W': 3, 'C': 576, 'k': 5,
                    'stride': 1, 'OH': 2, 'OW': 3, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 72, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 72, 'N': 2, 'H': 64, 'W': 128, 'C': 72, 'k': 5,
                    'stride': 2, 'OH': 32, 'OW': 64, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 672, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 672, 'N': 2, 'H': 16, 'W': 32, 'C': 672,
                    'k': 5, 'stride': 2, 'OH': 8, 'OW': 16, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 288, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 288, 'N': 2, 'H': 4, 'W': 6, 'C': 288, 'k': 5,
                    'stride': 2, 'OH': 2, 'OW': 3, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 96, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 96, 'N': 2, 'H': 8, 'W': 12, 'C': 96, 'k': 5,
                    'stride': 2, 'OH': 4, 'OW': 6, 'act': 0, 'gap_sum': None, 'op_dtype': 1}),
    ('dwconv_tma', {'x': 0, 'ldx': 16, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 16, 'N': 2, 'H': 128, 'W': 256, 'C': 16,
                    'k': 3, 'stride': 1, 'OH': 128, 'OW': 256, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 72, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 72, 'N': 2, 'H': 64, 'W': 128, 'C': 72, 'k': 3,
                    'stride': 1, 'OH': 64, 'OW': 128, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 200, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 200, 'N': 2, 'H': 16, 'W': 32, 'C': 200,
                    'k': 3, 'stride': 1, 'OH': 16, 'OW': 32, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 480, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 480, 'N': 2, 'H': 16, 'W': 32, 'C': 480,
                    'k': 3, 'stride': 1, 'OH': 16, 'OW': 32, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 88, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 88, 'N': 2, 'H': 8, 'W': 12, 'C': 88, 'k': 3,
                    'stride': 1, 'OH': 8, 'OW': 12, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 184, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 184, 'N': 2, 'H': 16, 'W': 32, 'C': 184,
                    'k': 3, 'stride': 1, 'OH': 16, 'OW': 32, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 256, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 256, 'N': 2, 'H': 8, 'W': 16, 'C': 256,
                    'k': 3, 'stride': 1, 'OH': 8, 'OW': 16, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 256, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 256, 'N': 2, 'H': 2, 'W': 3, 'C': 256, 'k': 3,
                    'stride': 1, 'OH': 2, 'OW': 3, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 16, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 16, 'N': 2, 'H': 32, 'W': 48, 'C': 16, 'k': 3,
                    'stride': 2, 'OH': 16, 'OW': 24, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 72, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 72, 'N': 2, 'H': 16, 'W': 24, 'C': 72, 'k': 3,
                    'stride': 2, 'OH': 8, 'OW': 12, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 240, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 240, 'N': 2, 'H': 32, 'W': 64, 'C': 240,
                    'k': 3, 'stride': 2, 'OH': 16, 'OW': 32, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 64, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 64, 'N': 2, 'H': 128, 'W': 256, 'C': 64,
                    'k': 3, 'stride': 2, 'OH': 64, 'OW': 128, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 144, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 144, 'N': 2, 'H': 4, 'W': 6, 'C': 144, 'k': 5,
                    'stride': 1, 'OH': 4, 'OW': 6, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 240, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 240, 'N': 2, 'H': 4, 'W': 6, 'C': 240, 'k': 5,
                    'stride': 1, 'OH': 4, 'OW': 6, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 120, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 120, 'N': 2, 'H': 32, 'W': 64, 'C': 120,
                    'k': 5, 'stride': 1, 'OH': 32, 'OW': 64, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 120, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 120, 'N': 2, 'H': 4, 'W': 6, 'C': 120, 'k': 5,
                    'stride': 1, 'OH': 4, 'OW': 6, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 960, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 960, 'N': 2, 'H': 8, 'W': 16, 'C': 960,
                    'k': 5, 'stride': 1, 'OH': 8, 'OW': 16, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 576, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 576, 'N': 2, 'H': 2, 'W': 3, 'C': 576, 'k': 5,
                    'stride': 1, 'OH': 2, 'OW': 3, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 72, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 72, 'N': 2, 'H': 64, 'W': 128, 'C': 72, 'k': 5,
                    'stride': 2, 'OH': 32, 'OW': 64, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 672, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 672, 'N': 2, 'H': 16, 'W': 32, 'C': 672,
                    'k': 5, 'stride': 2, 'OH': 8, 'OW': 16, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 288, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 288, 'N': 2, 'H': 4, 'W': 6, 'C': 288, 'k': 5,
                    'stride': 2, 'OH': 2, 'OW': 3, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('dwconv_tma', {'x': 0, 'ldx': 96, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 96, 'N': 2, 'H': 8, 'W': 12, 'C': 96, 'k': 5,
                    'stride': 2, 'OH': 4, 'OW': 6, 'act': 0, 'gap_sum': None, 'op_dtype': 2}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 128, 'Cin': 64, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 1,
                          'rows_pad': 128, 'k_pad': 64, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 16, 'Cin': 16, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 1,
                          'rows_pad': 16, 'k_pad': 64, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 24, 'Cin': 64, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 1,
                          'rows_pad': 32, 'k_pad': 64, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 72, 'Cin': 16, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 1,
                          'rows_pad': 80, 'k_pad': 64, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 64, 'Cin': 64, 'KH': 3, 'KW': 3, 'out': 0, 'out_dtype': 1,
                          'rows_pad': 64, 'k_pad': 64, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 64, 'Cin': 16, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 1,
                          'rows_pad': 16, 'k_pad': 64, 'transpose_flip': 1}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 16, 'Cin': 16, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 1,
                          'rows_pad': 16, 'k_pad': 64, 'transpose_flip': 1}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 24, 'Cin': 72, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 1,
                          'rows_pad': 80, 'k_pad': 64, 'transpose_flip': 1}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 256, 'Cin': 256, 'KH': 3, 'KW': 3, 'out': 0, 'out_dtype': 1,
                          'rows_pad': 256, 'k_pad': 256, 'transpose_flip': 1}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 128, 'Cin': 64, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 2,
                          'rows_pad': 128, 'k_pad': 64, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 16, 'Cin': 16, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 2,
                          'rows_pad': 16, 'k_pad': 64, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 24, 'Cin': 64, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 2,
                          'rows_pad': 32, 'k_pad': 64, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 72, 'Cin': 16, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 2,
                          'rows_pad': 80, 'k_pad': 64, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 64, 'Cin': 64, 'KH': 3, 'KW': 3, 'out': 0, 'out_dtype': 2,
                          'rows_pad': 64, 'k_pad': 64, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 64, 'Cin': 16, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 2,
                          'rows_pad': 16, 'k_pad': 64, 'transpose_flip': 1}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 16, 'Cin': 16, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 2,
                          'rows_pad': 16, 'k_pad': 64, 'transpose_flip': 1}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 24, 'Cin': 72, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 2,
                          'rows_pad': 80, 'k_pad': 64, 'transpose_flip': 1}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 256, 'Cin': 256, 'KH': 3, 'KW': 3, 'out': 0, 'out_dtype': 2,
                          'rows_pad': 256, 'k_pad': 256, 'transpose_flip': 1}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 16, 'Cin': 16, 'KH': 1, 'KW': 1, 'out': 0, 'out_dtype': 0,
                          'rows_pad': 16, 'k_pad': 16, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 16, 'Cin': 3, 'KH': 3, 'KW': 3, 'out': 0, 'out_dtype': 0, 'rows_pad': 16,
                          'k_pad': 3, 'transpose_flip': 0}),
    ('pack_conv_weight', {'w_oihw': 0, 'Cout': 64, 'Cin': 3, 'KH': 7, 'KW': 7, 'out': 0, 'out_dtype': 0, 'rows_pad': 64,
                          'k_pad': 3, 'transpose_flip': 0}),
    ('pack_conv_weight_parity', {'w_oihw': 0, 'Cout': 64, 'Cin': 64, 'K': 3, 'pad': 1, 'py': 0, 'px': 0, 'KH2': 1,
                                 'KW2': 1, 'pad2': 0, 'out': 0, 'rows_pad': 64, 'k_pad': 64, 'out_dtype': 1}),
    ('pack_conv_weight_parity', {'w_oihw': 0, 'Cout': 64, 'Cin': 64, 'K': 3, 'pad': 1, 'py': 0, 'px': 1, 'KH2': 1,
                                 'KW2': 2, 'pad2': 0, 'out': 0, 'rows_pad': 64, 'k_pad': 64, 'out_dtype': 1}),
    ('pack_conv_weight_parity', {'w_oihw': 0, 'Cout': 64, 'Cin': 64, 'K': 3, 'pad': 1, 'py': 1, 'px': 0, 'KH2': 2,
                                 'KW2': 1, 'pad2': 0, 'out': 0, 'rows_pad': 64, 'k_pad': 64, 'out_dtype': 1}),
    ('pack_conv_weight_parity', {'w_oihw': 0, 'Cout': 64, 'Cin': 64, 'K': 3, 'pad': 1, 'py': 1, 'px': 1, 'KH2': 2,
                                 'KW2': 2, 'pad2': 0, 'out': 0, 'rows_pad': 64, 'k_pad': 64, 'out_dtype': 1}),
    ('pack_conv_weight_parity', {'w_oihw': 0, 'Cout': 64, 'Cin': 64, 'K': 3, 'pad': 1, 'py': 0, 'px': 0, 'KH2': 1,
                                 'KW2': 1, 'pad2': 0, 'out': 0, 'rows_pad': 64, 'k_pad': 64, 'out_dtype': 2}),
    ('pack_conv_weight_parity', {'w_oihw': 0, 'Cout': 64, 'Cin': 64, 'K': 3, 'pad': 1, 'py': 0, 'px': 1, 'KH2': 1,
                                 'KW2': 2, 'pad2': 0, 'out': 0, 'rows_pad': 64, 'k_pad': 64, 'out_dtype': 2}),
    ('pack_conv_weight_parity', {'w_oihw': 0, 'Cout': 64, 'Cin': 64, 'K': 3, 'pad': 1, 'py': 1, 'px': 0, 'KH2': 2,
                                 'KW2': 1, 'pad2': 0, 'out': 0, 'rows_pad': 64, 'k_pad': 64, 'out_dtype': 2}),
    ('pack_conv_weight_parity', {'w_oihw': 0, 'Cout': 64, 'Cin': 64, 'K': 3, 'pad': 1, 'py': 1, 'px': 1, 'KH2': 2,
                                 'KW2': 2, 'pad2': 0, 'out': 0, 'rows_pad': 64, 'k_pad': 64, 'out_dtype': 2}),
    ('pack_dw_weight', {'w': 0, 'C': 16, 'k': 3, 'flip': 0, 'out': 0}),
    ('pack_dw_weight', {'w': 0, 'C': 16, 'k': 3, 'flip': 1, 'out': 0}),
    ('pack_dw_weight', {'w': 0, 'C': 72, 'k': 5, 'flip': 0, 'out': 0}),
    ('pack_dw_weight', {'w': 0, 'C': 120, 'k': 5, 'flip': 1, 'out': 0}),
    ('embed_filter', {'w_small': 0, 'Cout': 16, 'Cin': 3, 'k': 3, 'K': 7, 'w_big': 0, 'ld_big': 152, 'extract_add': 0}),
    ('embed_filter', {'w_small': 0, 'Cout': 16, 'Cin': 3, 'k': 3, 'K': 7, 'w_big': 0, 'ld_big': 152, 'extract_add': 1}),
    ('embed_filter', {'w_small': 0, 'Cout': 64, 'Cin': 3, 'k': 7, 'K': 7, 'w_big': 0, 'ld_big': 152, 'extract_add': 0}),
    ('embed_filter', {'w_small': 0, 'Cout': 64, 'Cin': 3, 'k': 7, 'K': 7, 'w_big': 0, 'ld_big': 152, 'extract_add': 1}),
    ('im2col_nchw', {'x': 0, 'N': 2, 'Cin': 3, 'H': 256, 'W': 512, 'k': 7, 'stride': 2, 'pad': 3, 'out': 0, 'ld': 152,
                     'out_dtype': 1}),
    ('im2col_nchw', {'x': 0, 'N': 2, 'Cin': 3, 'H': 64, 'W': 96, 'k': 7, 'stride': 2, 'pad': 3, 'out': 0, 'ld': 152,
                     'out_dtype': 1}),
    ('im2col_nchw', {'x': 0, 'N': 2, 'Cin': 3, 'H': 256, 'W': 512, 'k': 7, 'stride': 2, 'pad': 3, 'out': 0, 'ld': 152,
                     'out_dtype': 2}),
    ('im2col_nchw', {'x': 0, 'N': 2, 'Cin': 3, 'H': 64, 'W': 96, 'k': 7, 'stride': 2, 'pad': 3, 'out': 0, 'ld': 152,
                     'out_dtype': 2}),
    ('transpose_tokens', {'x': 0, 'ldx': 128, 'out': 0, 'N': 2, 'L': 128, 'C': 128, 'op_dtype': 1}),
    ('transpose_tokens', {'x': 0, 'ldx': 128, 'out': 0, 'N': 2, 'L': 128, 'C': 128, 'op_dtype': 2}),
    ('attn_softmax', {'s': 0, 'scale': 0.08838834764831845, 'p': 0, 'p_half': 0, 'rows': 256, 'cols': 128,
                      'op_dtype': 1}),
    ('attn_softmax', {'s': 0, 'scale': 0.08838834764831845, 'p': 0, 'p_half': 0, 'rows': 256, 'cols': 128,
                      'op_dtype': 2}),
    ('attn_softmax_backward', {'p': 0, 'dp': 0, 'ds_half': 0, 'rows': 256, 'cols': 128, 'alpha': 0.08838834764831845,
                               'op_dtype': 1}),
    ('attn_softmax_backward', {'p': 0, 'dp': 0, 'ds_half': 0, 'rows': 256, 'cols': 128, 'alpha': 0.08838834764831845,
                               'op_dtype': 2}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 1, 'sxn': 0, 'sxh': 0, 'sxw': 128, 'sxc': 1, 'x_batch_stride': 768, 'w': 0,
                     'w_dtype': 1, 'w_sco': 128, 'w_sk': 1, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 6, 'y_batch_stride': 36, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 128, 'Cout': 6, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 1, 'sxn': 0, 'sxh': 0, 'sxw': 128, 'sxc': 1, 'x_batch_stride': 768, 'w': 0,
                     'w_dtype': 1, 'w_sco': 128, 'w_sk': 1, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 6, 'y_batch_stride': 36, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 128, 'Cout': 6, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 0.08838834764831845}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 2, 'sxn': 0, 'sxh': 0, 'sxw': 128, 'sxc': 1, 'x_batch_stride': 768, 'w': 0,
                     'w_dtype': 2, 'w_sco': 128, 'w_sk': 1, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 6, 'y_batch_stride': 36, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 128, 'Cout': 6, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 2, 'sxn': 0, 'sxh': 0, 'sxw': 128, 'sxc': 1, 'x_batch_stride': 768, 'w': 0,
                     'w_dtype': 2, 'w_sco': 128, 'w_sk': 1, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 6, 'y_batch_stride': 36, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 128, 'Cout': 6, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 0.08838834764831845}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 0, 'sxh': 0, 'sxw': 6, 'sxc': 1, 'x_batch_stride': 36, 'w': 0,
                     'w_dtype': 1, 'w_sco': 1, 'w_sk': 128, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 128, 'y_batch_stride': 768, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 6, 'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 0, 'sxh': 0, 'sxw': 1, 'sxc': 6, 'x_batch_stride': 36, 'w': 0,
                     'w_dtype': 1, 'w_sco': 1, 'w_sk': 128, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 1, 'ldy': 128, 'y_batch_stride': 768, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 6, 'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 0, 'sxh': 0, 'sxw': 6, 'sxc': 1, 'x_batch_stride': 36, 'w': 0,
                     'w_dtype': 2, 'w_sco': 1, 'w_sk': 128, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 128, 'y_batch_stride': 768, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 6, 'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 0, 'sxh': 0, 'sxw': 1, 'sxc': 6, 'x_batch_stride': 36, 'w': 0,
                     'w_dtype': 2, 'w_sco': 1, 'w_sk': 128, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 2, 'ldy': 128, 'y_batch_stride': 768, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 6, 'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 0, 'sxh': 0, 'sxw': 6, 'sxc': 1, 'x_batch_stride': 36, 'w': 0,
                     'w_dtype': 0, 'w_sco': 1, 'w_sk': 128, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 128, 'y_batch_stride': 768, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 6, 'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 0, 'sxh': 0, 'sxw': 128, 'sxc': 1, 'x_batch_stride': 768, 'w': 0,
                     'w_dtype': 0, 'w_sco': 128, 'w_sk': 1, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 6, 'y_batch_stride': 36, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 128, 'Cout': 6, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 0, 'sxh': 0, 'sxw': 128, 'sxc': 1, 'x_batch_stride': 768, 'w': 0,
                     'w_dtype': 0, 'w_sco': 128, 'w_sk': 1, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 6, 'y_batch_stride': 36, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 128, 'Cout': 6, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 0.08838834764831845}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 0, 'sxh': 0, 'sxw': 1, 'sxc': 6, 'x_batch_stride': 36, 'w': 0,
                     'w_dtype': 0, 'w_sco': 1, 'w_sk': 128, 'w_batch_stride': 768, 'bias': None, 'res': None,
                     'ldres': 0, 'y': 0, 'y_dtype': 0, 'ldy': 128, 'y_batch_stride': 768, 'batches': 2, 'N': 1, 'H': 1,
                     'W': 6, 'Cin': 6, 'Cout': 128, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 1, 'OW': 6, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 1536, 'sxh': 768, 'sxw': 256, 'sxc': 1, 'x_batch_stride': 0, 'w': 0,
                     'w_dtype': 0, 'w_sco': 256, 'w_sk': 1, 'w_batch_stride': 0, 'bias': 0, 'res': None, 'ldres': 0,
                     'y': 0, 'y_dtype': 0, 'ldy': 8, 'y_batch_stride': 0, 'batches': 1, 'N': 2, 'H': 2, 'W': 3,
                     'Cin': 256, 'Cout': 8, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 2, 'OW': 3, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 2304, 'sxh': 576, 'sxw': 96, 'sxc': 1, 'x_batch_stride': 0, 'w': 0,
                     'w_dtype': 0, 'w_sco': 96, 'w_sk': 1, 'w_batch_stride': 0, 'bias': None, 'res': None, 'ldres': 0,
                     'y': 0, 'y_dtype': 0, 'ldy': 40, 'y_batch_stride': 0, 'batches': 1, 'N': 2, 'H': 4, 'W': 6,
                     'Cin': 96, 'Cout': 40, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 4, 'OW': 6, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 4992, 'sxh': 2496, 'sxw': 832, 'sxc': 1, 'x_batch_stride': 0, 'w': 0,
                     'w_dtype': 0, 'w_sco': 7488, 'w_sk': 1, 'w_batch_stride': 0, 'bias': None, 'res': None, 'ldres': 0,
                     'y': 0, 'y_dtype': 0, 'ldy': 256, 'y_batch_stride': 0, 'batches': 1, 'N': 2, 'H': 2, 'W': 3,
                     'Cin': 832, 'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'OH': 2, 'OW': 3, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 24576, 'sxh': 1536, 'sxw': 64, 'sxc': 1, 'x_batch_stride': 0, 'w': 0,
                     'w_dtype': 0, 'w_sco': 576, 'w_sk': 1, 'w_batch_stride': 0, 'bias': None, 'res': None, 'ldres': 0,
                     'y': 0, 'y_dtype': 0, 'ldy': 64, 'y_batch_stride': 0, 'batches': 1, 'N': 2, 'H': 16, 'W': 24,
                     'Cin': 64, 'Cout': 64, 'KH': 3, 'KW': 3, 'stride': 2, 'pad': 1, 'OH': 8, 'OW': 12, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 4992, 'sxh': 2496, 'sxw': 832, 'sxc': 1, 'x_batch_stride': 0, 'w': 0,
                     'w_dtype': 0, 'w_sco': 256, 'w_sk': 1, 'w_batch_stride': 0, 'bias': 0, 'res': None, 'ldres': 0,
                     'y': 0, 'y_dtype': 0, 'ldy': 256, 'y_batch_stride': 0, 'batches': 1, 'N': 2, 'H': 2, 'W': 3,
                     'Cin': 256, 'Cout': 256, 'KH': 1, 'KW': 1, 'stride': 1, 'pad': 0, 'OH': 2, 'OW': 3, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 4992, 'sxh': 2496, 'sxw': 832, 'sxc': 1, 'x_batch_stride': 0, 'w': 0,
                     'w_dtype': 0, 'w_sco': 5184, 'w_sk': 1, 'w_batch_stride': 0, 'bias': None, 'res': None, 'ldres': 0,
                     'y': 0, 'y_dtype': 0, 'ldy': 256, 'y_batch_stride': 0, 'batches': 1, 'N': 2, 'H': 2, 'W': 3,
                     'Cin': 576, 'Cout': 256, 'KH': 3, 'KW': 3, 'stride': 1, 'pad': 1, 'OH': 2, 'OW': 3, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 18432, 'sxh': 96, 'sxw': 1, 'sxc': 6144, 'x_batch_stride': 0, 'w': 0,
                     'w_dtype': 0, 'w_sco': 27, 'w_sk': 1, 'w_batch_stride': 0, 'bias': None, 'res': None, 'ldres': 0,
                     'y': 0, 'y_dtype': 0, 'ldy': 16, 'y_batch_stride': 0, 'batches': 1, 'N': 2, 'H': 64, 'W': 96,
                     'Cin': 3, 'Cout': 16, 'KH': 3, 'KW': 3, 'stride': 2, 'pad': 1, 'OH': 32, 'OW': 48, 'act': 0,
                     'alpha': 1.0}),
    ('conv2d_simt', {'x': 0, 'x_dtype': 0, 'sxn': 18432, 'sxh': 96, 'sxw': 1, 'sxc': 6144, 'x_batch_stride': 0, 'w': 0,
                     'w_dtype': 0, 'w_sco': 147, 'w_sk': 1, 'w_batch_stride': 0, 'bias': None, 'res': None, 'ldres': 0,
                     'y': 0, 'y_dtype': 0, 'ldy': 64, 'y_batch_stride': 0, 'batches': 1, 'N': 2, 'H': 64, 'W': 96,
                     'Cin': 3, 'Cout': 64, 'KH': 7, 'KW': 7, 'stride': 2, 'pad': 3, 'OH': 32, 'OW': 48, 'act': 0,
                     'alpha': 1.0}),
    ('dwconv', {'x': 0, 'ldx': 256, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 256, 'dtype': 0, 'N': 2, 'H': 2, 'W': 3, 'C': 256,
                'k': 3, 'stride': 1, 'OH': 2, 'OW': 3, 'act': 0, 'gap_sum': None}),
    ('dwconv', {'x': 0, 'ldx': 16, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 16, 'dtype': 0, 'N': 2, 'H': 32, 'W': 48, 'C': 16,
                'k': 3, 'stride': 2, 'OH': 16, 'OW': 24, 'act': 0, 'gap_sum': None}),
    ('dwconv', {'x': 0, 'ldx': 120, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 120, 'dtype': 0, 'N': 2, 'H': 4, 'W': 6, 'C': 120,
                'k': 5, 'stride': 1, 'OH': 4, 'OW': 6, 'act': 0, 'gap_sum': None}),
    ('dwconv', {'x': 0, 'ldx': 288, 'w': 0, 'bias': 0, 'y': 0, 'ldy': 288, 'dtype': 0, 'N': 2, 'H': 4, 'W': 6, 'C': 288,
                'k': 5, 'stride': 2, 'OH': 2, 'OW': 3, 'act': 0, 'gap_sum': None}),
    ('gate_fc', {'in': 0, 'in_scale': 0.00048828125, 'W': 0, 'b': None, 'out': 0, 'N': 2, 'C': 256, 'J': 64, 'act': 1,
                 'in_fixed': 0}),
    ('gate_fc', {'in': 0, 'in_scale': 0.0026041666666666665, 'W': 0, 'b': 0, 'out': 0, 'N': 2, 'C': 16, 'J': 8,
                 'act': 1, 'in_fixed': 0}),
    ('gate_fc', {'in': 0, 'in_scale': 1.0, 'W': 0, 'b': 0, 'out': 0, 'N': 2, 'C': 8, 'J': 16, 'act': 3, 'in_fixed': 0}),
    ('gate_fc', {'in': 0, 'in_scale': 1.0, 'W': 0, 'b': None, 'out': 0, 'N': 2, 'C': 64, 'J': 256, 'act': 4,
                 'in_fixed': 0}),
    ('cab_combine', {'g': 0, 'x': 0, 'r': 0, 'out': 0, 'ldo': 832, 'gamma': 0, 'dtype': 1, 'n_pixels': 12, 'C': 256}),
    ('cab_combine', {'g': 0, 'x': 0, 'r': 0, 'out': 0, 'ldo': 832, 'gamma': 0, 'dtype': 2, 'n_pixels': 12, 'C': 256}),
    ('cab_combine', {'g': 0, 'x': 0, 'r': 0, 'out': 0, 'ldo': 832, 'gamma': 0, 'dtype': 0, 'n_pixels': 12, 'C': 256}),
    ('softmax_rows', {'s': 0, 'p': 0, 'p_dtype': 0, 'rows': 256, 'cols': 128}),
    ('softmax_rows', {'s': 0, 'p': 0, 'p_dtype': 0, 'rows': 12, 'cols': 6}),
    ('upsample_logits_nchw', {'x': 0, 'N': 2, 'IH': 8, 'IW': 12, 'C': 8, 'y': 0, 'y_dtype': 0, 'OH': 64, 'OW': 96}),
    ('bn_frozen_stats', {'gamma': 0, 'beta': 0, 'running_mean': 0, 'running_var': 0, 'eps': 1e-05, 'C': 16,
                         'stats': 0}),
]


@pytest.mark.parametrize("entry,a", [pytest.param(e, a, id=variant_key(e, a).replace(" ", "_")) for e, a in CASES])
def test_variant_against_float64(entry, a):
    lib = _lib.load()
    k = Case()
    k.keep = []
    call = RUNNERS[entry](lib, a, k)
    first = _launch(lib, k, call, entry)
    for name, op, ref, how in k.checks:
        check(f"{entry} {name}", op, ref, how)
    again = _launch(lib, k, call, entry)
    for b0, b1 in zip(first, again):
        assert torch.equal(b0.view(ITD[b0.dtype]), b1.view(ITD[b1.dtype])), f"{entry}: not bit-reproducible"

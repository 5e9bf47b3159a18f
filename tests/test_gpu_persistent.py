"""GPU: the persistent inference kernels walked past their first tile, at the tile counts the bench forward runs them with.

One case per production plan key (tests/persistent_plans.py).  Each case
  * runs the kernel twice on a batch whose outputs are channel windows (ld > C, offset 8) of NaN-filled buffers: the two
    runs must be bit-identical, no NaN may remain in the window and the neighbouring channels must keep their NaN bits;
  * runs every image of the batch alone (another CTA-to-tile mapping): the same bits as in the batch;
  * compares every output element with a float64 reference of the same op, computed per image on the device with the
    kernel's bf16 roundings, within a bound derived from magnitudes: ``2^-16 * mag + 1 ulp`` of the output, where
    ``mag`` is the same chain of ops on |inputs| and |weights|; a bf16 rounding inside a fused block may flip by one ulp,
    and that ulp is carried through the absolute weights of the ops behind it;
  * checks int64 fixed-point pooling sums (2^-24) per (image, channel) against the float64 sums, and across runs.
"""

import pytest
import torch
import torch.nn.functional as F

from tests import persistent_plans as pp

pytestmark = pytest.mark.gpu

from cabinet_b200 import _lib  # noqa: E402
from cabinet_b200._lib import ACT_HSWISH, ACT_NONE, ACT_RELU, check  # noqa: E402
from tests.test_gpu_ops import _pack_aux, _pack_aux_t, _pack_expand, _pack_expand_t, _pack_tc  # noqa: E402

OFF, EXTRA = 8, 24            # output windows: channels [8, 8 + C) of C + 24
NAN16, NAN32 = 0x7FC1, 0x7FC00001
LIP = {ACT_NONE: 1.0, ACT_RELU: 1.0, ACT_HSWISH: 1.5}   # Lipschitz bound of each activation (hard-swish: 1.5 at x = 3)
D = torch.float64


def stream():
    return torch.cuda.current_stream().cuda_stream


def act(x, a):
    if a == ACT_RELU:
        return F.relu(x)
    if a == ACT_HSWISH:
        return x * F.relu6(x + 3) / 6
    assert a == ACT_NONE
    return x


def bf(x):
    return x.to(torch.bfloat16).to(D)


def ulp(x, dtype=torch.bfloat16):
    """one unit in the last place of each element of x (already in `dtype`'s grid), as float64; 0 at 0."""
    _, e = torch.frexp(x.float())
    u = torch.ldexp(torch.ones_like(x, dtype=D), e.to(D).sub(8 if dtype == torch.bfloat16 else 24))
    return torch.where(x == 0, torch.zeros_like(u), u)


def cpu_gen(*shape, seed, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale


def dev_gen(*shape, seed, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator(device="cuda").manual_seed(seed), device="cuda") * scale


def conv(x, w, s=1, p=0, groups=1):
    """float64 convolution of one image; dense ones as a GEMM over unfolded patches."""
    if groups > 1:
        return F.conv2d(x, w, None, s, p, 1, groups)
    O, C, kh, kw = w.shape
    OH, OW = (x.shape[2] + 2 * p - kh) // s + 1, (x.shape[3] + 2 * p - kw) // s + 1
    cols = x.reshape(C, -1) if (kh, kw, s, p) == (1, 1, 1, 0) else F.unfold(x, (kh, kw), padding=p, stride=s)[0]
    return (w.reshape(O, -1) @ cols).view(1, O, OH, OW)


def window(N, H, W, C, dtype=torch.bfloat16):
    t = torch.empty((N, H, W, C + EXTRA), dtype=dtype, device="cuda")
    t.view(torch.int16 if dtype == torch.bfloat16 else torch.int32).fill_(NAN16 if dtype == torch.bfloat16 else NAN32)
    return t


def inputs(N, H, W, C, seed):
    """bf16 NHWC activations in channels [OFF, OFF + C) of a wider buffer (as the engine's concat slices)."""
    t = torch.zeros((N, H, W, C + 16), dtype=torch.bfloat16, device="cuda")
    t[..., OFF:OFF + C] = dev_gen(N, H, W, C, seed=seed).to(torch.bfloat16)
    return t


def nchw(t, n, C):
    return t[n:n + 1, ..., OFF:OFF + C].permute(0, 3, 1, 2).to(D)


def ptr(t, n=0, C=0):
    """address of image n, channel OFF (C > 0) or channel 0 of a batched buffer."""
    return t.data_ptr() + n * t[0].numel() * t.element_size() + (OFF * t.element_size() if C else 0)


def check_windows(buf, C):
    bits = buf.view(torch.int16 if buf.dtype == torch.bfloat16 else torch.int32)
    nan = NAN16 if buf.dtype == torch.bfloat16 else NAN32
    assert not torch.isnan(buf[..., OFF:OFF + C]).any(), "a tile was not written"
    assert bool((bits[..., :OFF] == nan).all()) and bool((bits[..., OFF + C:] == nan).all()), "neighbouring channels written"


def compare(case, plan, n, got, ref, bound):
    """got / ref / bound: [1, C, OH, OW] float64.  -> worst err / bound; fails with the tile of the first bad element."""
    err = (got - ref).abs()
    bad = err > bound
    if bool(bad.any()):
        i = bad.nonzero()[0].tolist()
        th, tw = plan.get("TH", 1), plan.get("TW", 1)
        raise AssertionError(f"{case['id']}: {int(bad.sum())} elements out of bound; first: image {n} channel {i[1]} "
                             f"pixel ({i[2]}, {i[3]}) = tile ({i[2] // th}, {i[3] // tw}), got {float(got[tuple(i)])}, "
                             f"want {float(ref[tuple(i)])} +- {float(bound[tuple(i)])}")
    return float((err / bound).max())


def compare_sums(case, n, got_fixed, ref, bound):
    got = got_fixed.to(D) * 2.0 ** -24
    err = (got - ref).abs()
    assert bool((err <= bound).all()), f"{case['id']}: pooling sums of image {n}: worst {float((err / bound).max()):.3g} x bound"
    return float((err / bound).max())


# ------------------------------------------------------------------------------------------------ the kernels
class Mbconv:
    """mbconv_t / mbconv_fused in project, squeeze-excite-gated project, or depthwise-output (+ pooling sums) mode."""

    def __init__(self, c):
        self.c, self.fused = c, c["entry"] == "mbconv_fused"
        cin, cexp, cout, k = c["Cin"], c["Cexp"], c["Cout"], c["k"]
        self.mode = "se" if c.get("se_scale") else ("project" if c["w_project"] else "dw")
        self.cy = cout if self.mode != "dw" else cexp
        self.x = inputs(c["N"], c["H"], c["W"], cin, seed=1)
        self.we, self.be = bf(cpu_gen(cexp, cin, 1, 1, seed=2, scale=cin ** -0.5)), cpu_gen(cexp, seed=3, scale=0.2)
        self.wd, self.bd = cpu_gen(cexp, 1, k, k, seed=4, scale=1.0 / k), cpu_gen(cexp, seed=5, scale=0.1)
        if self.fused:
            self.pe, self.aux = _pack_expand(self.we.float(), self.be), _pack_aux(self.wd, self.be, self.bd)
        else:
            self.pe, self.aux = _pack_expand_t(self.we.float(), self.be), _pack_aux_t(self.wd, self.bd)
        if self.mode != "dw":
            self.wp, self.bp = bf(cpu_gen(cout, cexp, 1, 1, seed=6, scale=cexp ** -0.5)), cpu_gen(cout, seed=7, scale=0.1)
            self.pp, self.bpd = _pack_tc(self.wp.float()), self.bp.cuda()
        self.gate = torch.rand((c["N"], cexp), generator=torch.Generator().manual_seed(8)).cuda() if self.mode == "se" else None
        self.dev = {k_: v.to("cuda", D) for k_, v in (("we", self.we), ("be", self.be), ("wd", self.wd), ("bd", self.bd))}
        if self.mode != "dw":
            self.dev.update(wp=self.wp.to("cuda", D), bp=self.bp.to("cuda", D))

    def launch(self, n0, N):
        c = self.c
        y = window(N, c["OH"], c["OW"], self.cy)
        gap = torch.zeros((N, c["Cexp"]), dtype=torch.int64, device="cuda") if self.mode == "dw" else None
        fn = _lib.load().cabinet_mbconv_fused if self.fused else _lib.load().cabinet_mbconv_t
        project = self.mode != "dw"
        args = [ptr(self.x, n0, 1), self.x.shape[-1], N, c["H"], c["W"], c["Cin"], self.pe.data_ptr(), self.aux.data_ptr(),
                c["Cexp"], c["act_expand"], c["k"], c["stride"], c["act_dw"], self.pp.data_ptr() if project else None,
                self.bpd.data_ptr() if project else None, c["Cout"] if project else 0, c["residual"], ptr(y, 0, 1),
                y.shape[-1], c["OH"], c["OW"], gap.data_ptr() if gap is not None else None]
        if not self.fused:
            args.append(self.gate[n0].data_ptr() if self.gate is not None else None)
        check(fn(*args, stream()), c["entry"])
        return y, gap

    def reference(self, n):
        c, d = self.c, self.dev
        k, s, pad = c["k"], c["stride"], (c["k"] - 1) // 2
        x = nchw(self.x, n, c["Cin"])
        h = conv(x, d["we"]) + d["be"].view(1, -1, 1, 1)
        mh = conv(x.abs(), d["we"].abs()) + d["be"].abs().view(1, -1, 1, 1)
        a, ma, ea = act(h, c["act_expand"]), LIP[c["act_expand"]] * mh, 0.0
        if self.fused:  # the pixel-major kernel stages the expanded activation as bf16
            a = bf(a)
            ea = ulp(a)
        pre = conv(a, d["wd"], s, pad, c["Cexp"]) + d["bd"].view(1, -1, 1, 1)
        mpre = conv(ma, d["wd"].abs(), s, pad, c["Cexp"]) + d["bd"].abs().view(1, -1, 1, 1)
        epre = conv(ea, d["wd"].abs(), s, pad, c["Cexp"]) if self.fused else torch.zeros_like(pre)
        lip = LIP[c["act_dw"]]
        if self.mode == "dw":
            out = bf(act(pre, c["act_dw"]))
            bound = 2.0 ** -16 * lip * mpre + lip * epre + ulp(out)
            return out, bound, pre.sum((2, 3))[0], 2.0 ** -16 * (mpre + epre).sum((2, 3))[0]
        g = self.gate[n].to(D).view(1, -1, 1, 1) if self.gate is not None else 1.0
        dq = bf(act(pre * g, c["act_dw"]))
        md, ed = lip * g * mpre, lip * g * epre + ulp(dq)
        y = conv(dq, d["wp"]) + d["bp"].view(1, -1, 1, 1)
        my = conv(md, d["wp"].abs()) + d["bp"].abs().view(1, -1, 1, 1)
        if c["residual"]:
            y, my = y + x, my + x.abs()
        y = bf(y)
        return y, 2.0 ** -16 * my + conv(ed, d["wp"].abs()) + ulp(y), None, None


class Stem:
    """stem_tc2: sb.conv1 (7x7 s2, ReLU) and the mobile stem (3x3 s2, hard-swish) of the fp32 NCHW image."""

    def __init__(self, c):
        self.c = c
        self.x = dev_gen(c["N"], 3, c["H"], c["W"], seed=1)
        w7, b7 = cpu_gen(64, 3, 7, 7, seed=2, scale=0.1), cpu_gen(64, seed=3, scale=0.1)
        w3, b3 = cpu_gen(16, 3, 3, 3, seed=4, scale=0.2), cpu_gen(16, seed=5, scale=0.1)
        pk = torch.zeros(80, 3, 7, 8)
        pk[:64, :, :, 1:8] = w7
        pk[64:, :, 2:5, 3:6] = w3
        bias = torch.cat([b7, b3])
        wn = torch.zeros(80, 7, 8, 4)               # W[o][ky][kx][c]; c = 3 is the constant-1 channel
        wn[..., :3] = pk.permute(0, 2, 3, 1)
        hi = bias.to(torch.bfloat16).float()
        wn[:, 3, 4, 3], wn[:, 3, 5, 3] = hi, bias - hi
        self.wk = wn.view(80, 7, 2, 2, 8).permute(1, 2, 3, 0, 4).contiguous().to("cuda", torch.bfloat16)
        self.w7, self.w3 = bf(w7).cuda(), bf(w3).cuda()
        self.b7, self.b3 = b7.to("cuda", D), b3.to("cuda", D)

    def launch(self, n0, N):
        c = self.c
        sb, st = window(N, c["OH"], c["OW"], 64), window(N, c["OH"], c["OW"], 16)
        check(_lib.load().cabinet_stem_tc2(self.x[n0].data_ptr(), N, c["H"], c["W"], self.wk.data_ptr(), ptr(sb, 0, 1),
                                           sb.shape[-1], ptr(st, 0, 1), st.shape[-1], c["OH"], c["OW"], stream()), "stem_tc2")
        return (sb, st), None

    def reference(self, n):
        x = bf(self.x[n:n + 1].to(D))
        outs, bounds = [], []
        for w, b, p, a in ((self.w7, self.b7, 3, ACT_RELU), (self.w3, self.b3, 1, ACT_HSWISH)):
            y = bf(act(conv(x, w, 2, p) + b.view(1, -1, 1, 1), a))
            mag = conv(x.abs(), w.abs(), 2, p) + b.abs().view(1, -1, 1, 1)
            outs.append(y)
            bounds.append(2.0 ** -16 * LIP[a] * mag + ulp(y))
        return outs, bounds, None, None


class ExpandSums:
    """expand_sums with the automatic split: pooling sums of the depthwise BN output of a squeeze-excite block."""

    def __init__(self, c):
        self.c = c
        self.m = Mbconv(dict(c, entry="mbconv_t", Cout=0, stride=1, act_dw=ACT_NONE, OH=c["H"], OW=c["W"], residual=0,
                             w_project=None, se_scale=None))

    def launch(self, n0, N):
        c, m = self.c, self.m
        gap = torch.zeros((N, c["Cexp"]), dtype=torch.int64, device="cuda")
        check(_lib.load().cabinet_expand_sums(ptr(m.x, n0, 1), m.x.shape[-1], N, c["H"], c["W"], c["Cin"], m.pe.data_ptr(),
                                              m.aux.data_ptr(), c["Cexp"], c["act_expand"], c["k"], c["nsplit"],
                                              gap.data_ptr(), stream()), "expand_sums")
        return None, gap

    def reference(self, n):
        _, _, s, b = self.m.reference(n)
        return None, None, s, b


class ConvTc:
    """conv_tc_se (with and without the squeeze-excite prologue), conv_tc_imgw (per-image weights), conv_tc_split_act."""

    def __init__(self, c):
        self.c = c
        N, cin, cout, k = c["N"], c["Cin"], c["Cout"], c["KH"]
        self.f32 = c["y_dtype"] == 0
        self.x = inputs(N, c["H"], c["W"], cin, seed=1)
        self.res = inputs(N, c["OH"], c["OW"], cout, seed=9) if c.get("res") else None
        self.scale = torch.rand((N, cin), generator=torch.Generator().manual_seed(5)).cuda() if c.get("a_scale") else None
        nw = N if c["entry"] == "conv_tc_imgw" else 1
        self.w = [bf(cpu_gen(cout, cin, k, k, seed=10 + i, scale=(cin * k * k) ** -0.5)) for i in range(nw)]
        self.b = cpu_gen(cout, seed=3, scale=0.3)
        n16, c64 = -(-cout // 16) * 16, -(-cin // 64) * 64
        pk = torch.zeros(nw, n16, k * k, c64)
        for i, w in enumerate(self.w):
            pk[i, :cout, :, :cin] = w.float().permute(0, 2, 3, 1).reshape(cout, k * k, cin)
        self.pk, self.wstride = pk.to("cuda", torch.bfloat16).contiguous(), n16 * k * k * c64
        self.bd, self.wdev = self.b.cuda(), [w.cuda() for w in self.w]

    def launch(self, n0, N):
        c, lib = self.c, _lib.load()
        y = window(N, c["OH"], c["OW"], c["Cout"], torch.float32 if self.f32 else torch.bfloat16)
        # fp32 outputs take any channel offset: 3
        yp, ldy = y.data_ptr() + (3 if self.f32 else OFF) * y.element_size(), y.shape[-1]
        res = (ptr(self.res, n0, 1), self.res.shape[-1]) if self.res is not None else (None, 0)
        geo = (c["Cout"], c["KH"], c["KW"], c["stride"], c["pad"])
        if c["entry"] == "conv_tc_imgw":
            check(lib.cabinet_conv_tc_imgw(ptr(self.x, n0, 1), self.x.shape[-1], N, c["H"], c["W"], c["Cin"],
                                           self.pk[n0].data_ptr(), self.wstride, *geo, self.bd.data_ptr(), *res, yp,
                                           c["y_dtype"], ldy, c["OH"], c["OW"], c["act"], stream()), "conv_tc_imgw")
        elif c["entry"] == "conv_tc_split_act":
            check(lib.cabinet_conv_tc_split_act(ptr(self.x, n0, 1), self.x.shape[-1], N, c["H"], c["W"], c["Cin"],
                                                self.pk.data_ptr(), *geo, self.bd.data_ptr(), yp, c["y_dtype"], ldy, c["OH"],
                                                c["OW"], c["act"], c["act_cols"], stream()), "conv_tc_split_act")
        else:
            check(lib.cabinet_conv_tc_se(ptr(self.x, n0, 1), self.x.shape[-1], N, c["H"], c["W"], c["Cin"],
                                         self.scale[n0].data_ptr() if self.scale is not None else None, c["a_act"],
                                         self.pk.data_ptr(), *geo, self.bd.data_ptr(), *res, yp, c["y_dtype"], ldy,
                                         c["OH"], c["OW"], c["act"], stream()), "conv_tc_se")
        return y, None

    def reference(self, n):
        c = self.c
        x = nchw(self.x, n, c["Cin"])
        w = self.wdev[n if len(self.wdev) > 1 else 0].to(D)
        ea = None
        if self.scale is not None:  # the prologue re-rounds act(x * s) to bf16 in shared memory: one ulp may flip
            x = bf(act(x * self.scale[n].to(D).view(1, -1, 1, 1), c["a_act"]))
            ea = ulp(x)
        b = self.bd.to(D).view(1, -1, 1, 1)
        z = conv(x, w, c["stride"], c["pad"]) + b
        mag = conv(x.abs(), w.abs(), c["stride"], c["pad"]) + b.abs()
        if ea is not None:
            mag = mag + 2.0 ** 16 * conv(ea, w.abs(), c["stride"], c["pad"])
        if self.res is not None:
            r = nchw(self.res, n, c["Cout"])
            z, mag = z + r, mag + r.abs()
        cols = c.get("act_cols", c["Cout"])
        y = torch.cat([act(z[:, :cols], c["act"]), z[:, cols:]], 1)
        lip = LIP[c["act"]]
        y = y if self.f32 else bf(y)
        return y, 2.0 ** -16 * lip * mag + ulp(y, torch.float32 if self.f32 else torch.bfloat16), None, None


RUNNERS = {"mbconv_t": Mbconv, "mbconv_fused": Mbconv, "stem_tc2": Stem, "expand_sums": ExpandSums, "conv_tc_se": ConvTc,
           "conv_tc_imgw": ConvTc, "conv_tc_split_act": ConvTc}


def _outputs(y):
    return [] if y is None else (list(y) if isinstance(y, tuple) else [y])


def _channels(t, f32):
    off = 3 if f32 else OFF
    return off, t.shape[-1] - EXTRA


@pytest.mark.parametrize("case", pp.CASES, ids=[c["id"] for c in pp.CASES])
def test_persistent_walk(case):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    plan = pp.case_plan(case, sms)
    k = RUNNERS[case["entry"]](case)
    N = case["N"]
    y1, g1 = k.launch(0, N)
    y2, g2 = k.launch(0, N)
    torch.cuda.synchronize()
    outs1, outs2 = _outputs(y1), _outputs(y2)
    for a, b in zip(outs1, outs2):
        assert torch.equal(a.view(torch.int16), b.view(torch.int16)), "two runs differ"
        f32 = a.dtype == torch.float32
        off, C = _channels(a, f32)
        if f32:
            bits = a.view(torch.int32)
            assert not torch.isnan(a[..., off:off + C]).any(), "a tile was not written"
            assert bool((bits[..., :off] == NAN32).all()) and bool((bits[..., off + C:] == NAN32).all())
        else:
            check_windows(a, C)
    if g1 is not None:
        assert torch.equal(g1, g2), "pooling sums differ between runs"
    if case["entry"] != "expand_sums":  # its automatic split depends on the batch: each image alone is another plan
        for n in range(N):
            yn, gn = k.launch(n, 1)
            torch.cuda.synchronize()
            for a, b in zip(outs1, _outputs(yn)):
                assert torch.equal(a[n:n + 1].view(torch.int16), b.view(torch.int16)), f"image {n} alone differs from the batch"
            if g1 is not None:
                assert torch.equal(g1[n:n + 1], gn), f"pooling sums of image {n} alone differ from the batch"
            del yn, gn
    worst, worst_sum = 0.0, 0.0
    for n in range(N):
        ref, bound, rsum, bsum = k.reference(n)
        refs, bounds = (ref, bound) if isinstance(ref, list) else ([ref] if ref is not None else [], [bound])
        for a, r, bd in zip(outs1, refs, bounds):
            off, C = _channels(a, a.dtype == torch.float32)
            got = a[n:n + 1, ..., off:off + C].permute(0, 3, 1, 2).to(D)
            worst = max(worst, compare(case, plan, n, got, r, bd))
        if rsum is not None:
            # each contribution to an int64 accumulator is rounded to 2^-24 once: one per tile and thread segment
            worst_sum = max(worst_sum, compare_sums(case, n, g1[n], rsum, bsum + 16 * plan["tiles_img"] * 2.0 ** -24))
        del ref, bound
    print(f"{case['id']}: {plan['tiles']} tiles, grid {plan['grid']}, {plan['per_cta']:.2f} tiles per CTA, "
          f"worst err / bound {worst:.3f}" + (f", sums {worst_sum:.3f}" if g1 is not None else ""))

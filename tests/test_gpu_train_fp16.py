"""GPU: the fp16 training mode (``model.train_precision = "fp16"``) -- the reference's autocast + GradScaler numerics.

* per kernel: the bf16 cases of ``test_gpu_train.py`` repeated with fp16 activations (fp32 torch on the same fp16-rounded
  inputs; fp16 output rounding, 2^-11 relative, in place of bf16's 2^-8), the tensor-core / staging kernels through their
  ``*_dt`` entry points;
* the whole step against the reference's OWN fp16 noise: ``oracle.train_oracle.train_step`` under
  ``torch.autocast("cuda", dtype=torch.float16)`` (what ``train.py`` does to the reference model) vs the fp32 oracle;
* graph replay bit-identical to the eager schedule, and ``torch.amp.GradScaler`` skipping an overflowing step.
"""

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from cabinet_b200 import _lib  # noqa: E402
from cabinet_b200._lib import F16, check  # noqa: E402
from cabinet_b200.constants import BACKBONE_CFGS  # noqa: E402
from cabinet_b200.loss import OhemCELoss  # noqa: E402
from cabinet_b200.synthetic import build_model, make_input, make_labels  # noqa: E402
from cabinet_b200.train_engine import TrainEngine  # noqa: E402
from oracle.train_oracle import train_step  # noqa: E402
from tests import test_gpu_train as T  # noqa: E402
from tests.gpu_util import rel_l2  # noqa: E402

H16 = torch.float16
FP16_TOL = 100.0   # fp16 outputs: 2^-11 relative rounding per element (bf16: 400 for 2^-9)


@pytest.fixture(autouse=True)
def fp16_tables(monkeypatch):
    """The dtype tables of the bf16 cases, extended by fp16 for the duration of a test."""
    monkeypatch.setitem(T.DT, H16, F16)
    monkeypatch.setitem(T.TOLS, H16, FP16_TOL)


def params_of(fn):
    """The parameter sets of a test of test_gpu_train.py (its dtype axis dropped): the fp16 cases are the same ones."""
    out, names = [], None
    for mark in reversed(fn.pytestmark):
        if mark.name != "parametrize" or mark.args[0] == "dtype":
            continue
        names, out = mark.args[0], list(mark.args[1])
    return names, out


@pytest.mark.parametrize(*params_of(T.test_bn_train_forward_backward))
def test_bn_train_forward_backward_fp16(N, C, H, W, act):
    T.test_bn_train_forward_backward(N, C, H, W, act, H16)


@pytest.mark.parametrize(*params_of(T.test_conv_gradients))
def test_conv_gradients_fp16(N, cin, cout, k, s, p, H, W, nchw_in):
    T.test_conv_gradients(N, cin, cout, k, s, p, H, W, nchw_in, H16)


@pytest.mark.parametrize(*params_of(T.test_dwconv_gradients))
def test_dwconv_gradients_fp16(N, C, k, s, H, W):
    T.test_dwconv_gradients(N, C, k, s, H, W, H16)


@pytest.mark.parametrize(*params_of(T.test_gate_backward))
def test_gate_backward_fp16(gate, plus, act, bias):
    T.test_gate_backward(gate, plus, act, bias, H16)


@pytest.mark.parametrize(*params_of(T.test_resample_band_kernel_x8_adjoint))
def test_resample_band_kernel_x8_adjoint_fp16(h, w):
    T.test_resample_band_kernel_x8_adjoint(h, w, H16)


@pytest.mark.parametrize(*params_of(T.test_conv_wgrad_tensor_core))
def test_conv_wgrad_tensor_core_fp16(N, cin, cout, k, H, W, ldx_extra, stride):
    lib = _lib.load()
    p = (k - 1) // 2
    x = T.q(T.gen(N, cin, H, W, seed=1), H16)
    w = T.gen(cout, cin, k, k, seed=2, scale=0.1).requires_grad_(True)
    y = F.conv2d(x, w, None, stride, p)
    dy = T.q(T.gen(*y.shape, seed=3), H16)
    y.backward(dy)
    ldx = cin + ldx_extra
    xb = torch.zeros(N, H, W, ldx, dtype=H16, device="cuda")
    xb[..., ldx_extra:] = T.nhwc(x, H16)
    xv = xb[..., ldx_extra:]
    dyd = T.nhwc(dy, H16)
    n = int(lib.cabinet_conv_wgrad_tc_scratch_floats(N, H, W, cin, cout, k, k, stride, p))
    sc = torch.full((n,), float("nan"), device="cuda")
    dw = torch.zeros(cout, cin, k, k, device="cuda")
    check(lib.cabinet_conv_wgrad_tc_dt(dyd.data_ptr(), cout, xv.data_ptr(), ldx, dw.data_ptr(), N, H, W, cin, cout, k, k,
                                       stride, p, sc.data_ptr(), F16, T.stream()), "wgrad_tc_dt")
    torch.cuda.synchronize()
    assert rel_l2(dw.cpu(), w.grad) < 1e-5   # exact products of fp16 values, fp32 accumulation


@pytest.mark.parametrize(*params_of(T.test_stride2_dgrad_as_parity_conv_tc))
def test_stride2_dgrad_as_parity_conv_tc_fp16(N, cin, cout, k, pad, H, W):
    lib = _lib.load()
    x = T.gen(N, cin, H, W, seed=1).requires_grad_(True)
    w = T.q(T.gen(cout, cin, k, k, seed=2, scale=(cin * k * k) ** -0.5), H16).requires_grad_(True)
    y = F.conv2d(x, w, None, 2, pad)
    dy = T.q(T.gen(*y.shape, seed=3), H16)
    y.backward(dy)
    OH, OW = y.shape[2:]
    dyd, wd = T.nhwc(dy, H16), w.detach().cuda()
    dx = torch.full((N, H, W, cin), 5.0, dtype=H16, device="cuda")
    zeros = torch.zeros(cin, device="cuda")
    r16, k64 = -(-cin // 16) * 16, -(-cout // 64) * 64
    for py in range(2):
        for px in range(2):
            (kh2, pad2), (kw2, _) = TrainEngine._parity_geom(k, pad, py), TrainEngine._parity_geom(k, pad, px)
            hc, wc = (H - py + 1) // 2, (W - px + 1) // 2
            wt = torch.empty(r16, kh2 * kw2, k64, dtype=H16, device="cuda")
            check(lib.cabinet_pack_conv_weight_parity_dt(wd.data_ptr(), cout, cin, k, pad, py, px, kh2, kw2, pad2,
                                                         wt.data_ptr(), r16, k64, F16, T.stream()), "pack_parity_dt")
            check(lib.cabinet_conv_tc_view_dt(dyd.data_ptr(), cout, N, OH, OW, cout, wt.data_ptr(), cin, kh2, kw2, pad2,
                                              zeros.data_ptr(), dx.data_ptr() + (py * W + px) * cin * 2, cin, hc, wc, 2, 2 * W,
                                              H * W, F16, T.stream()), "conv_tc_view_dt")
    torch.cuda.synchronize()
    assert rel_l2(T.nchw(dx), x.grad) < 1e-3   # fp16 output rounding (bf16: 4e-3)


@pytest.mark.parametrize(*params_of(T.test_stem_im2col_and_embedded_filter))
def test_stem_im2col_fp16(N, H, W):
    lib = _lib.load()
    x = T.gen(N, 3, H, W, seed=1)
    OH, OW, LD = (H - 1) // 2 + 1, (W - 1) // 2 + 1, 152
    col = torch.full((N * OH * OW, LD), 9.0, dtype=H16, device="cuda")
    check(lib.cabinet_im2col_nchw_dt(x.cuda().data_ptr(), N, 3, H, W, 7, 2, 3, col.data_ptr(), LD, F16, T.stream()), "im2col")
    ref = F.unfold(x.to(H16).float(), 7, padding=3, stride=2).transpose(1, 2).reshape(N * OH * OW, 147)
    torch.cuda.synchronize()
    assert torch.equal(col[:, :147].float().cpu(), ref) and float(col[:, 147:].abs().max()) == 0


def test_conv_tc_fp16_forward_and_overflow():
    """conv_tc with fp16 operands against fp32 torch on the same fp16 values (ReLU epilogue, residual), and an fp16
    overflow stays inf (round to nearest, never saturated)."""
    lib = _lib.load()
    N, cin, cout, H, W = 2, 64, 96, 12, 20
    x = T.q(T.gen(N, cin, H, W, seed=1), H16)
    w = T.q(T.gen(cout, cin, 3, 3, seed=2, scale=(cin * 9) ** -0.5), H16)
    res = T.q(T.gen(N, cout, H, W, seed=3), H16)
    r16, k64 = -(-cout // 16) * 16, -(-cin // 64) * 64
    wp = torch.empty(r16, 9, k64, dtype=H16, device="cuda")
    check(lib.cabinet_pack_conv_weight(w.cuda().data_ptr(), cout, cin, 3, 3, wp.data_ptr(), F16, r16, k64, 0, T.stream()), "pack")
    xd, rd, zb = T.nhwc(x, H16), T.nhwc(res, H16), torch.zeros(cout, device="cuda")
    ref = F.conv2d(x, w, None, 1, 1)
    for act, use_res in ((T.ACT_RELU, False), (T.ACT_NONE, True)):
        y = torch.empty(N, H, W, cout, dtype=H16, device="cuda")
        check(lib.cabinet_conv_tc_dt(xd.data_ptr(), cin, N, H, W, cin, wp.data_ptr(), cout, 3, 3, 1, 1, zb.data_ptr(),
                                     rd.data_ptr() if use_res else None, cout if use_res else 0, y.data_ptr(), F16, cout, H, W,
                                     act, F16, T.stream()), "conv_tc_dt")
        torch.cuda.synchronize()
        assert rel_l2(T.nchw(y), T.act_ref(ref, act) + (res if use_res else 0)) < 1e-3
    # weights x 1e5 (still finite in fp16): outputs of |y| ~ 1e5 > 65504 must come out as inf, not clamped
    wbig = T.q(w * 1e5, H16)
    check(lib.cabinet_pack_conv_weight(wbig.cuda().data_ptr(), cout, cin, 3, 3, wp.data_ptr(), F16, r16, k64, 0, T.stream()),
          "pack")
    y = torch.empty(N, H, W, cout, dtype=H16, device="cuda")
    check(lib.cabinet_conv_tc_dt(xd.data_ptr(), cin, N, H, W, cin, wp.data_ptr(), cout, 3, 3, 1, 1, zb.data_ptr(), None, 0,
                                 y.data_ptr(), F16, cout, H, W, T.ACT_RELU, F16, T.stream()), "conv_tc_dt")
    torch.cuda.synchronize()
    ref_big = F.relu(F.conv2d(x, wbig, None, 1, 1))
    big, yy = ref_big > 70000, T.nchw(y)
    assert bool(big.any()) and torch.isinf(yy[big]).all()
    assert rel_l2(yy[ref_big < 60000], ref_big[ref_big < 60000]) < 1e-3


def test_transpose_tokens_and_attn_softmax_fp16():
    lib = _lib.load()
    N, L, C, ld = 3, 70, 40, 48
    x = T.gen(N, L, ld, seed=4).cuda().to(H16)
    out = torch.empty(N, C, L, device="cuda", dtype=H16)
    check(lib.cabinet_transpose_tokens_dt(x.data_ptr(), ld, out.data_ptr(), N, L, C, F16, T.stream()), "transpose_tokens")
    assert torch.equal(out, x[:, :, :C].transpose(1, 2).contiguous())
    rows, cols = 37, 130
    s = T.gen(rows, cols, seed=5, scale=4.0).cuda()
    p, p16 = torch.empty_like(s), torch.empty(rows, cols, device="cuda", dtype=H16)
    check(lib.cabinet_attn_softmax_dt(s.data_ptr(), 0.37, p.data_ptr(), p16.data_ptr(), rows, cols, F16, T.stream()), "softmax")
    assert rel_l2(p, torch.softmax(s * 0.37, dim=-1)) < 1e-6 and torch.equal(p16, p.to(H16))
    dp = T.gen(rows, cols, seed=6).cuda()
    ds = torch.empty(rows, cols, device="cuda", dtype=H16)
    check(lib.cabinet_attn_softmax_backward_dt(p.data_ptr(), dp.data_ptr(), ds.data_ptr(), rows, cols, 0.37, F16, T.stream()),
          "softmax_bwd")
    torch.cuda.synchronize()
    assert torch.equal(ds, (p * (dp - (dp * p).sum(-1, keepdim=True)) * 0.37).to(H16))


def test_conv_wgrad_tc_batched_fp16():
    lib = _lib.load()
    N, H, W, cin, cout = 3, 8, 16, 128, 200
    a = T.gen(N, H * W, cout, seed=7).cuda().to(H16)
    x = T.gen(N, H * W, cin, seed=8).cuda().to(H16)
    out = torch.full((N, cout, cin), 7.0, device="cuda")
    check(lib.cabinet_conv_wgrad_tc_batched_dt(a.data_ptr(), cout, x.data_ptr(), cin, out.data_ptr(), N, H, W, cin, cout, F16,
                                               T.stream()), "wgrad_batched_dt")
    torch.cuda.synchronize()
    assert rel_l2(out, torch.einsum("npo,npi->noi", a.float(), x.float())) < 1e-5


# ---------------------------------------------------------------------------------------------------- the whole step
def _step(model, x, lb, thresh, n_min):
    model.zero_grad(set_to_none=True)
    loss, _, _ = T._run_step(model, x, lb, thresh, n_min)
    named = dict(model.named_parameters())
    return loss, {k: p.grad.clone() for k, p in named.items() if p.grad is not None}, model.state_dict()


@pytest.mark.parametrize("mode,C,N,H,W", [("large", 6, 2, 96, 80), ("small", 8, 2, 64, 96)])
def test_train_step_fp16_vs_the_reference_autocast_noise(mode, C, N, H, W):
    """Every gradient, the loss and the running statistics of the fp16 mode against the fp32 oracle, within 1.25 x the
    deviation of the oracle itself under torch.autocast(fp16) + 0.01; the fp16 mode's median gradient error below the
    bf16 mode's (fp16 storage is in use); two fp16 runs bit-identical."""
    thresh, n_min = 0.7, N * H * W // 16
    base = build_model(C, mode)
    sd = {k: v.clone() for k, v in base.state_dict().items()}
    x, lb = make_input(N, H, W), make_labels(N, H, W, C)
    cfgs = BACKBONE_CFGS[mode]
    loss_ref, grads_ref, running_ref = train_step(sd, x, lb, cfgs, thresh, n_min)
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    with torch.autocast("cuda", dtype=torch.float16):
        loss_ac, grads_ac, running_ac = train_step(sd_gpu, x.cuda(), lb.cuda(), cfgs, thresh, n_min)
    typical = float(torch.tensor([float(g.norm()) for g in grads_ref.values() if g is not None]).median())
    errs, runs = {}, []
    for precision in ("fp16", "fp16", "bf16"):
        model = build_model(C, mode).cuda().train()
        model.train_precision = precision
        loss, grads, msd = _step(model, x.cuda(), lb.cuda(), thresh, n_min)
        runs.append(grads)
        e_all = []
        for k, gr in grads_ref.items():
            if gr is None:
                assert k not in grads
                continue
            e = rel_l2(grads[k].cpu(), gr)
            e_all.append(e)
            if precision != "fp16":
                continue
            bar = 1.25 * rel_l2(grads_ac[k].float().cpu(), gr) + 0.01
            small = float((grads[k].cpu() - gr).norm()) < 1e-1 * typical   # analytically ~0 gradients
            assert e <= bar or small, (k, e, bar)
        errs[precision] = float(torch.tensor(e_all).median())
        if precision == "fp16":
            bar = 1.25 * abs(float(loss_ac) - float(loss_ref)) / abs(float(loss_ref)) + 0.01
            assert abs(float(loss) - float(loss_ref)) / abs(float(loss_ref)) <= bar
            for prefix, (rm, rv) in running_ref.items():
                am, av = running_ac[prefix]
                assert rel_l2(msd[prefix + ".running_mean"].cpu(), rm) <= 1.25 * rel_l2(am.float().cpu(), rm) + 0.01, prefix
                assert rel_l2(msd[prefix + ".running_var"].cpu(), rv) <= 1.25 * rel_l2(av.float().cpu(), rv) + 0.01, prefix
    print(f"{mode}: median gradient rel_l2 fp16 {errs['fp16']:.3e}, bf16 {errs['bf16']:.3e}")
    assert errs["fp16"] < errs["bf16"]
    assert runs[0].keys() == runs[1].keys() and all(torch.equal(runs[0][k], runs[1][k]) for k in runs[0])


def test_train_step_graph_replay_is_bit_identical_to_eager_fp16():
    T.test_train_step_graph_replay_is_bit_identical_to_eager("fp16")


@pytest.mark.parametrize("init_scale,overflow", [(2.0 ** 16, False), (2.0 ** 40, True)])
def test_grad_scaler_fp16(init_scale, overflow):
    """torch.amp.GradScaler over the fp16 step, past the graph capture: at the default scale every gradient is finite and
    the parameters move; at 2^40 the fp16 data gradients overflow, the inf reaches the parameter gradients and
    ``scaler.step`` skips the step (parameters bit-identical, scale halved) in the eager AND the replayed steps."""
    C, N, H, W = 8, 2, 64, 96
    model = build_model(C, "small").cuda().train()
    model.train_precision = "fp16"
    opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9)
    scaler = torch.amp.GradScaler("cuda", init_scale=init_scale)
    crit = OhemCELoss(0.7, N * H * W // 16, 255)
    eng = model.train_engine()
    for step in range(5):
        x, lb = make_input(N, H, W, seed=step).cuda(), make_labels(N, H, W, C, seed=step).cuda()
        before = [p.detach().clone() for p in model.parameters()]
        opt.zero_grad(set_to_none=True)
        out, out16 = model(x)
        loss = crit(out, lb) + crit(out16, lb)
        scale = scaler.get_scale()
        scaler.scale(loss).backward()
        scaler.unscale_(opt)
        torch.nn.utils.clip_grad_norm_(model.parameters(), 10.0)
        scaler.step(opt)
        scaler.update()
        grads = [p.grad for p in model.parameters() if p.grad is not None]
        finite = all(bool(torch.isfinite(g).all()) for g in grads)
        same = all(torch.equal(a, p.detach()) for a, p in zip(before, model.parameters()))
        replayed = any(st.fwd is not None for st in eng._gsteps.values())
        if overflow:
            assert not finite and same and scaler.get_scale() == scale / 2, (step, replayed)
        else:
            assert finite and not same and scaler.get_scale() == scale, (step, replayed)
    assert replayed   # the last steps ran on the captured graphs

"""GPU: partial fine-tuning in the training step -- parameters with ``requires_grad=False`` and BatchNorm modules in eval
mode inside a ``.train()`` model, with PyTorch's semantics.

* ``cabinet_bn_frozen_stats`` / ``cabinet_bn_frozen_backward`` against eval-mode ``F.batch_norm`` + activation under
  autograd (fp32, bf16, fp16; dense, ragged C, pixel stride > C, accumulate), running statistics untouched, bit-
  reproducible, nothing written past the documented scratch size (a canary block behind it, one-block reductions
  included); the parameter-only form over batch statistics against train-mode autograd;
* whole fp32 steps against the oracle with the same modules frozen: all BN eval, backbone frozen, heads only, and a mix
  (eval BN with trainable gamma / beta, a train-mode BN behind a frozen convolution); frozen ``p.grad`` stays ``None``
  and an SGD step leaves frozen parameters and frozen BN buffers bit-identical;
* bf16 / fp16 steps with all BN eval, ``GradScaler`` over a frozen backbone in fp16;
* graph replay bit-identical to the eager schedule while the backbone is frozen and unfrozen mid-run.
"""

import pytest
import torch
import torch.nn.functional as F
from torch import nn

pytestmark = pytest.mark.gpu

from cabinet_b200 import _lib  # noqa: E402
from cabinet_b200._lib import ACT_HSWISH, ACT_NONE, ACT_RELU, BF16, F16, F32, check  # noqa: E402
from cabinet_b200.constants import BACKBONE_CFGS  # noqa: E402
from cabinet_b200.loss import OhemCELoss  # noqa: E402
from cabinet_b200.synthetic import build_model, make_input, make_labels  # noqa: E402
from oracle import cabinet_oracle  # noqa: E402
from oracle.loss_oracle import ohem_ce_loss  # noqa: E402
from tests.gpu_util import rel_l2  # noqa: E402
from tests.test_gpu_train import act_ref, gen, nchw, q, scratch, stream  # noqa: E402

DT = {torch.float32: F32, torch.bfloat16: BF16, torch.float16: F16}
TOLS = {torch.float32: 1.0, torch.bfloat16: 400.0, torch.float16: 100.0}   # 2^-9 / 2^-11 relative rounding per element
SHAPES = [(2, 16, 9, 7, ACT_RELU), (3, 72, 5, 5, ACT_HSWISH), (1, 960, 2, 2, ACT_NONE), (2, 300, 17, 13, ACT_RELU),
          (4, 64, 96, 97, ACT_RELU), (2, 120, 80, 73, ACT_HSWISH), (1, 960, 41, 40, ACT_NONE), (3, 16, 160, 150, ACT_HSWISH)]


KINKS = {ACT_RELU: (0.0,), ACT_HSWISH: (-3.0, 3.0), ACT_NONE: ()}


def _off_kinks(x, gamma, beta, act, dtype, rm=None, rv=None):
    """x moved (by 1/16, exact in every dtype here) wherever the BN output u lies within 1e-3 of a kink of the
    activation's derivative: there act'(u) is decided by the last bit of u, which the kernel (z * scale + shift) and
    F.batch_norm ((z - mean) * invstd * gamma + beta) round differently."""
    x = x.detach().clone()
    for _ in range(4):
        with torch.no_grad():
            u = F.batch_norm(x, rm, rv, gamma, beta, rm is None, 0.0, 1e-5)
        near = torch.zeros_like(x, dtype=torch.bool)
        for k in KINKS[act]:
            near |= (u - k).abs() < 1e-3
        if not near.any():
            return q(x, dtype)
        x[near] += 0.0625
    raise AssertionError("could not move the inputs off the activation's kinks")


CANARY = 4096   # floats after the documented scratch size: a write past the end lands here


def _scratch(lib, M, C, nq, canaries):
    """Scratch of exactly the documented size (M, C, nq), followed by a canary block the test checks afterwards."""
    n = int(lib.cabinet_train_scratch_floats(M, C, nq))
    t = torch.full((n + CANARY,), -7.0, device="cuda")
    canaries.append(t[n:])
    return t


def _padded(t_nchw, dtype, ld):
    """NCHW cpu -> NHWC cuda with pixel stride ``ld`` >= C (a channel slice of a wider buffer)."""
    N, C, H, W = t_nchw.shape
    buf = torch.full((N, H, W, ld), float("nan"), dtype=dtype, device="cuda")
    buf[..., :C] = t_nchw.permute(0, 2, 3, 1).to(dtype).cuda()
    return buf


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("N,C,H,W,act,extra,acc", [s + (0, 0) for s in SHAPES] + [
    (2, 13, 11, 9, ACT_RELU, 0, 0),        # ragged C: the scalar kernels
    (2, 64, 24, 20, ACT_HSWISH, 8, 0),     # pixel stride > C, still vector aligned
    (2, 40, 15, 17, ACT_RELU, 3, 0),       # pixel stride > C, unaligned: scalar
    (3, 72, 30, 30, ACT_HSWISH, 0, 1),     # accumulate into dz
    (2, 30, 12, 12, ACT_NONE, 5, 1)])
def test_bn_frozen_forward_backward(N, C, H, W, act, extra, acc, dtype):
    lib = _lib.load()
    dt, tm = DT[dtype], TOLS[dtype]
    gamma, beta = (gen(C, seed=2) * 0.3 + 1).requires_grad_(True), gen(C, seed=3, scale=0.2).requires_grad_(True)
    rm, rv = gen(C, seed=4, scale=0.5) + 5, gen(C, seed=5).abs() * 4 + 0.5
    x = _off_kinks(q(gen(N, C, H, W, seed=1) * 2 + 5, dtype), gamma, beta, act, dtype, rm, rv).requires_grad_(True)
    y_ref = act_ref(F.batch_norm(x, rm, rv, gamma, beta, False, 0.1, 1e-5), act)
    dy = q(gen(N, C, H, W, seed=6), dtype)
    y_ref.backward(dy)
    dz0 = q(gen(N, C, H, W, seed=7), dtype)   # what dz holds before an accumulating call
    M, ld = N * H * W, C + extra
    xd, dyd = _padded(x.detach(), dtype, ld), _padded(dy, dtype, ld)
    rmd, rvd, gd, bd = rm.cuda(), rv.cuda(), gamma.detach().cuda(), beta.detach().cuda()
    rm0, rv0 = rmd.clone(), rvd.clone()
    stats = torch.empty(4, C, device="cuda")
    check(lib.cabinet_bn_frozen_stats(gd.data_ptr(), bd.data_ptr(), rmd.data_ptr(), rvd.data_ptr(), 1e-5, C,
                                      stats.data_ptr(), stream()), "frozen_stats")
    y = _padded(torch.zeros(N, C, H, W), dtype, ld)
    check(lib.cabinet_affine_act(xd.data_ptr(), ld, dt, stats[2].data_ptr(), stats[3].data_ptr(), None, 0.0, None, 0,
                                 y.data_ptr(), ld, dt, M, H * W, C, act, stream()), "affine_act")

    canaries = []

    def backward():
        dz = _padded(dz0, dtype, ld)
        dg, db = torch.full((C,), 0.25, device="cuda"), torch.full((C,), -0.5, device="cuda")   # accumulated into
        check(lib.cabinet_bn_frozen_backward(dyd.data_ptr(), ld, xd.data_ptr(), ld, dt, stats.data_ptr(), act,
                                             dg.data_ptr(), db.data_ptr(), dz.data_ptr(), ld, M, C, acc,
                                             _scratch(lib, M, C, 2, canaries).data_ptr(), stream()), "frozen_backward")
        return dz, dg, db

    dz, dg, db = backward()
    dz2, dg2, db2 = backward()
    # the two partial forms: data gradient only, parameter gradients only
    dz_only = _padded(dz0, dtype, ld)
    check(lib.cabinet_bn_frozen_backward(dyd.data_ptr(), ld, xd.data_ptr(), ld, dt, stats.data_ptr(), act, None, None,
                                         dz_only.data_ptr(), ld, M, C, acc, None, stream()), "frozen_backward dz")
    dg3, db3 = torch.full((C,), 0.25, device="cuda"), torch.full((C,), -0.5, device="cuda")
    check(lib.cabinet_bn_frozen_backward(dyd.data_ptr(), ld, xd.data_ptr(), ld, dt, stats.data_ptr(), act,
                                         dg3.data_ptr(), db3.data_ptr(), None, 0, M, C, 0,
                                         _scratch(lib, M, C, 2, canaries).data_ptr(), stream()), "frozen_backward params")
    torch.cuda.synchronize()
    assert all(bool((c == -7.0).all()) for c in canaries)   # nothing written past the documented scratch size
    assert torch.equal(rmd, rm0) and torch.equal(rvd, rv0)   # running statistics: bitwise untouched
    assert rel_l2(nchw(y[..., :C]), y_ref.detach()) < 1e-5 * tm
    dz_ref = x.grad + (dz0 if acc else 0)
    assert rel_l2(nchw(dz[..., :C]), dz_ref) < 1e-4 * tm / 4
    assert rel_l2(dg.cpu() - 0.25, gamma.grad) < 1e-4 and rel_l2(db.cpu() + 0.5, beta.grad) < 1e-4
    for t in (dz, dz_only):
        assert torch.isnan(t[..., C:]).all()   # nothing written outside the channel slice
    dz, dz2, dz_only = dz[..., :C], dz2[..., :C], dz_only[..., :C]
    assert torch.equal(dz, dz2) and torch.equal(dg, dg2) and torch.equal(db, db2)   # bit-reproducible
    assert torch.equal(dz, dz_only) and torch.equal(dg, dg3) and torch.equal(db, db3)   # the partial forms: same bits


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("N,C,H,W,act", [(2, 16, 9, 7, ACT_RELU), (2, 300, 17, 13, ACT_RELU), (4, 64, 96, 97, ACT_HSWISH)])
def test_bn_frozen_backward_gives_train_bn_parameter_gradients(N, C, H, W, act, dtype):
    """Batch statistics of cabinet_bn_train_stats + cabinet_bn_frozen_backward without dz: the gamma / beta gradients of a
    train-mode BN whose input needs no gradient."""
    lib = _lib.load()
    dt = DT[dtype]
    gamma, beta = (gen(C, seed=2) * 0.3 + 1).requires_grad_(True), gen(C, seed=3, scale=0.2).requires_grad_(True)
    x = _off_kinks(q(gen(N, C, H, W, seed=1) * 2 + 5, dtype), gamma, beta, act, dtype)
    y_ref = act_ref(F.batch_norm(x, None, None, gamma, beta, True, 0.1, 1e-5), act)
    dy = q(gen(N, C, H, W, seed=6), dtype)
    y_ref.backward(dy)
    M = N * H * W
    xd, dyd = _padded(x, dtype, C), _padded(dy, dtype, C)
    stats = torch.empty(4, C, device="cuda")
    gd, bd = gamma.detach().cuda(), beta.detach().cuda()
    check(lib.cabinet_bn_train_stats(xd.data_ptr(), C, dt, M, C, gd.data_ptr(), bd.data_ptr(), 1e-5, 0.1, None, None,
                                     stats.data_ptr(), scratch(lib, M, C, 2).data_ptr(), stream()), "stats")
    dg, db = torch.zeros(C, device="cuda"), torch.zeros(C, device="cuda")
    canaries = []
    check(lib.cabinet_bn_frozen_backward(dyd.data_ptr(), C, xd.data_ptr(), C, dt, stats.data_ptr(), act, dg.data_ptr(),
                                         db.data_ptr(), None, 0, M, C, 0, _scratch(lib, M, C, 2, canaries).data_ptr(),
                                         stream()), "bwd")
    torch.cuda.synchronize()
    assert bool((canaries[0] == -7.0).all())
    assert rel_l2(dg.cpu(), gamma.grad) < 1e-4 and rel_l2(db.cpu(), beta.grad) < 1e-4


# ----------------------------------------------------------------------------- whole steps
def oracle_step(sd, x, labels, cfgs, thresh, n_min, frozen_bn=(), frozen_params=()):
    """oracle/train_oracle.train_step with the BN prefixes in ``frozen_bn`` in eval mode (running statistics) and the
    parameters in ``frozen_params`` without a gradient -> (loss, {param: grad or None}, {trained BN: running stats})."""
    params = {k: v.clone().requires_grad_(k not in frozen_params) for k, v in sd.items()
              if v.is_floating_point() and not k.endswith(("running_mean", "running_var"))}
    work = dict(sd)
    work.update(params)
    bn = cabinet_oracle.bn

    def bn_with_frozen(sd_, prefix, x_):
        if prefix not in frozen_bn:
            return bn(sd_, prefix, x_)
        saved, cabinet_oracle.BATCH_STATS = cabinet_oracle.BATCH_STATS, None
        try:
            return bn(sd_, prefix, x_)
        finally:
            cabinet_oracle.BATCH_STATS = saved

    cabinet_oracle.BATCH_STATS, cabinet_oracle.bn = {}, bn_with_frozen
    try:
        out, out16 = cabinet_oracle.cabinet_forward_graph(work, x.float(), cfgs)
        stats = cabinet_oracle.BATCH_STATS
    finally:
        cabinet_oracle.BATCH_STATS, cabinet_oracle.bn = None, bn
    loss = ohem_ce_loss(out, labels, thresh, n_min) + ohem_ce_loss(out16, labels, thresh, n_min)
    loss.backward()
    running = {p: (0.9 * sd[p + ".running_mean"] + 0.1 * m, 0.9 * sd[p + ".running_var"] + 0.1 * v)
               for p, (m, v, _) in stats.items()}
    return loss.detach(), {k: p.grad for k, p in params.items()}, running


def bn_prefixes(model, under=("",)):
    return [n for n, m in model.named_modules() if isinstance(m, nn.BatchNorm2d) and n.startswith(under)]


def all_bn_eval(model):
    return bn_prefixes(model), []


def backbone_frozen(model):
    return bn_prefixes(model, ("mobile",)), [n for n, _ in model.named_parameters() if n.startswith("mobile")]


def heads_only(model):
    heads = ("ffm", "conv_out")
    return (bn_prefixes(model, ("mobile", "sb", "ab")),
            [n for n, _ in model.named_parameters() if not n.startswith(heads)])


def mixed(model):
    """eval BNs with trainable gamma / beta in the spatial and attention branches; the backbone stem convolution frozen
    in front of its train-mode BN (parameter gradients over batch statistics, no data gradient)."""
    return bn_prefixes(model, ("sb", "ab")), ["mobile.features.0.0.weight", "ab.convb.weight", "sb.conv2.conv.weight"]


SETTINGS = {"all_bn_eval": all_bn_eval, "backbone_frozen": backbone_frozen, "heads_only": heads_only, "mixed": mixed}


def apply_setting(model, setting, train=True):
    frozen_bn, frozen_params = SETTINGS[setting](model)
    mods, named = dict(model.named_modules()), dict(model.named_parameters())
    for p in frozen_bn:
        mods[p].train(not train)
    for n in frozen_params:
        named[n].requires_grad_(not train)
    return frozen_bn, frozen_params


def _step(model, x, lb, thresh, n_min, scale=1.0):
    crit_p, crit_16 = OhemCELoss(thresh, n_min, 255), OhemCELoss(thresh, n_min, 255)
    out, out16 = model(x)
    loss = crit_p(out, lb) + crit_16(out16, lb)
    (loss * scale).backward()
    return loss.detach()


@pytest.mark.parametrize("setting", list(SETTINGS))
def test_train_step_with_frozen_modules_vs_oracle(setting):
    """fp32 step against the oracle with the same modules frozen (the bars of
    test_train_step_all_gradients_vs_oracle_and_determinism), then an SGD step: frozen parameters and frozen BN buffers
    bit-identical, trained BNs at the oracle's running statistics."""
    mode, C, N, H, W = "large", 6, 2, 96, 80
    thresh, n_min = 0.7, N * H * W // 16
    base = build_model(C, mode)
    sd = {k: v.clone() for k, v in base.state_dict().items()}
    x, lb = make_input(N, H, W), make_labels(N, H, W, C)
    frozen_bn, frozen_params = SETTINGS[setting](base)
    loss_ref, grads_ref, running_ref = oracle_step(sd, x, lb, BACKBONE_CFGS[mode], thresh, n_min, set(frozen_bn),
                                                   set(frozen_params))
    model = build_model(C, mode).cuda().train()
    model.train_precision = "fp32"
    apply_setting(model, setting)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    loss = _step(model, x.cuda(), lb.cuda(), thresh, n_min)
    assert float(loss) == pytest.approx(float(loss_ref), rel=2e-4)
    named = dict(model.named_parameters())
    typical = float(torch.tensor([float(g.norm()) for g in grads_ref.values() if g is not None]).median())
    worst = ("", 0.0)
    for k, gr in grads_ref.items():
        if gr is None:
            assert named[k].grad is None, k   # frozen, or not on the forward path (mobile.classifier)
            continue
        e = rel_l2(named[k].grad.cpu(), gr)
        small = float((named[k].grad.cpu() - gr).norm()) < 1e-5 * typical
        if e > worst[1] and not small:
            worst = (k, e)
        assert e < 3e-2 or small, (setting, k, e)
    print(f"{setting}: loss {float(loss):.6f} vs {float(loss_ref):.6f}; worst gradient {worst[0]} rel_l2 {worst[1]:.2e}")
    torch.optim.SGD(model.parameters(), lr=0.1, momentum=0.9).step()
    after = model.state_dict()
    for n in frozen_params:
        assert torch.equal(after[n], before[n]), n
    for p in frozen_bn:
        for b in ("running_mean", "running_var", "num_batches_tracked"):
            assert torch.equal(after[f"{p}.{b}"], before[f"{p}.{b}"]), (p, b)
    for p, (rm, rv) in running_ref.items():
        assert rel_l2(after[p + ".running_mean"].cpu(), rm) < 1e-4 and rel_l2(after[p + ".running_var"].cpu(), rv) < 1e-4, p
        assert int(after[p + ".num_batches_tracked"]) == 1
    assert set(running_ref) == set(bn_prefixes(model)) - set(frozen_bn)


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_train_step_all_bn_eval_half_precisions(precision):
    """bf16 / fp16 activations with every BN in eval mode, within the bar of the bf16 step (each gradient within its own
    norm of the fp32 oracle's, the layer next to the loss within 8 %).  The loss is scaled by 2^10 and the gradients
    unscaled, as GradScaler does: without it, the deep fp16 activation gradients would sit in fp16's subnormal range."""
    mode, C, N, H, W = "large", 6, 2, 96, 80
    thresh, n_min = 0.7, N * H * W // 16
    base = build_model(C, mode)
    sd = {k: v.clone() for k, v in base.state_dict().items()}
    x, lb = make_input(N, H, W), make_labels(N, H, W, C)
    loss_ref, grads_ref, _ = oracle_step(sd, x, lb, BACKBONE_CFGS[mode], thresh, n_min, set(bn_prefixes(base)))
    model = build_model(C, mode).cuda().train()
    model.train_precision = precision
    apply_setting(model, "all_bn_eval")
    before = {k: v.clone() for k, v in model.state_dict().items() if not k.endswith(("weight", "bias", "gamma"))}
    loss = _step(model, x.cuda(), lb.cuda(), thresh, n_min, scale=1024.0)
    assert float(loss) == pytest.approx(float(loss_ref), rel=2e-2)
    named = dict(model.named_parameters())
    for p in named.values():
        if p.grad is not None:
            p.grad /= 1024.0
    typical = float(torch.tensor([float(g.norm()) for g in grads_ref.values() if g is not None]).median())
    for k, gr in grads_ref.items():
        if gr is None:
            assert named[k].grad is None, k
            continue
        e = rel_l2(named[k].grad.cpu(), gr)
        assert e < 1.0 or float((named[k].grad.cpu() - gr).norm()) < 1e-1 * typical, (precision, k, e)
    assert rel_l2(named["conv_out.conv_out.weight"].grad.cpu(), grads_ref["conv_out.conv_out.weight"]) < 0.08
    sd_after = model.state_dict()
    for k, v in before.items():
        assert torch.equal(sd_after[k], v), k   # running statistics and num_batches_tracked of every BN


@pytest.mark.parametrize("init_scale,overflow", [(2.0 ** 16, False), (2.0 ** 40, True)])
def test_grad_scaler_fp16_frozen_backbone(init_scale, overflow):
    """GradScaler over the fp16 step with a frozen backbone, past the graph capture: at 2^16 the trainable parameters
    move, at 2^40 the overflow reaches their gradients and the step is skipped; the backbone never moves."""
    C, N, H, W = 8, 2, 64, 96
    model = build_model(C, "small").cuda().train()
    model.train_precision = "fp16"
    apply_setting(model, "backbone_frozen")
    trainable = [p for p in model.parameters() if p.requires_grad]
    backbone = [p.detach().clone() for p in model.mobile.parameters()]
    opt = torch.optim.SGD(trainable, lr=0.01, momentum=0.9)
    scaler = torch.amp.GradScaler("cuda", init_scale=init_scale)
    crit = OhemCELoss(0.7, N * H * W // 16, 255)
    eng = model.train_engine()
    for step in range(5):
        x, lb = make_input(N, H, W, seed=step).cuda(), make_labels(N, H, W, C, seed=step).cuda()
        before = [p.detach().clone() for p in trainable]
        opt.zero_grad(set_to_none=True)
        out, out16 = model(x)
        scale = scaler.get_scale()
        scaler.scale(crit(out, lb) + crit(out16, lb)).backward()
        scaler.unscale_(opt)
        scaler.step(opt)
        scaler.update()
        assert all(p.grad is None for p in model.mobile.parameters())
        finite = all(bool(torch.isfinite(p.grad).all()) for p in trainable)
        same = all(torch.equal(a, p.detach()) for a, p in zip(before, trainable))
        if overflow:
            assert not finite and same and scaler.get_scale() == scale / 2, step
        else:
            assert finite and not same and scaler.get_scale() == scale, step
    assert any(st.fwd is not None for st in eng._gsteps.values())   # the last steps replayed the captured graphs
    assert all(torch.equal(a, p) for a, p in zip(backbone, model.mobile.parameters()))


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_graph_replay_with_freezing_mid_run(precision):
    """Eager schedule against graph replay over an SGD run that freezes the backbone at step 4 and unfreezes it at step
    9: logits, loss, every gradient and all buffers bit for bit; each change re-captures (two eager steps, then a new
    graph), so a replay never runs a graph captured for the other setting."""
    C, N, H, W = 5, 2, 96, 64
    models = []
    for use_graph in (False, True):
        m = build_model(C, "small").cuda().train()
        m.train_precision = precision
        m.train_engine().use_graph = use_graph
        models.append((m, torch.optim.SGD(m.parameters(), lr=0.01, momentum=0.9)))
    crit = OhemCELoss(0.7, N * H * W // 16, 255)
    eng = models[1][0].train_engine()
    for step in range(13):
        x = make_input(N, H, W, seed=step).cuda()
        lb = make_labels(N, H, W, C, seed=step).cuda()
        if step in (4, 9):
            for m, _ in models:
                apply_setting(m, "backbone_frozen", train=step == 4)
        res = []
        for m, opt in models:
            opt.zero_grad(set_to_none=True)
            out, out16 = m(x)
            loss = crit(out, lb) + crit(out16, lb)
            loss.backward()
            res.append((out.detach().clone(), out16.detach().clone(), loss.detach().clone(),
                        {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}))
            opt.step()
        (o0, a0, l0, g0), (o1, a1, l1, g1) = res
        assert torch.equal(o0, o1) and torch.equal(a0, a1) and torch.equal(l0, l1), step
        assert g0.keys() == g1.keys()
        assert any(k.startswith("mobile") for k in g1) == (step < 4 or step >= 9), step
        for k in g0:
            assert torch.equal(g0[k], g1[k]), (step, k)
        captured = [st for st in eng._gsteps.values() if st.fwd is not None]
        assert bool(captured) == (step >= eng.graph_after and step not in (4, 5, 9, 10)), step
        sd0, sd1 = models[0][0].state_dict(), models[1][0].state_dict()
        for k in sd0:
            assert torch.equal(sd0[k], sd1[k]), (step, k)

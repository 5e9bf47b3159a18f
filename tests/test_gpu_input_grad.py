"""GPU: gradients with respect to the input image (``x.grad``) in train mode and through an eval-mode model.

* ``cabinet_stem_dgrad`` against float64 autograd of the two stem ``F.conv2d`` calls on the same rounded dy and weights:
  fp32 / bf16 / fp16, even and odd sizes down to 1 x 1, either gradient NULL, padded pixel strides; NaN-prefilled output
  with canary margins, an elementwise bound, two runs bit-identical;
* the same train steps with and without ``x.requires_grad``: bit-identical logits, loss, gradients, running statistics;
* ``x.grad`` against the oracle (``oracle/cabinet_oracle.py`` under autograd): train mode fp32, eval mode fp32 with
  frozen parameters, the auxiliary output alone, bf16 / fp16 within the oracle's own autocast noise;
* composition with an upstream module, fp16 and channels_last inputs;
* graph replay: an eval-mode PGD loop and an adversarial-training loop bit-identical to the eager schedule.
"""

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from cabinet_b200 import _lib  # noqa: E402
from cabinet_b200._lib import BF16, F16, F32, check  # noqa: E402
from cabinet_b200.constants import BACKBONE_CFGS  # noqa: E402
from cabinet_b200.loss import OhemCELoss  # noqa: E402
from cabinet_b200.synthetic import build_model, make_input, make_labels  # noqa: E402
from oracle import cabinet_oracle  # noqa: E402
from oracle.loss_oracle import ohem_ce_loss  # noqa: E402
from tests.gpu_util import rel_l2  # noqa: E402
from tests.test_gpu_train import gen, stream  # noqa: E402

TORCH_DT = {F32: torch.float32, BF16: torch.bfloat16, F16: torch.float16}


# ----------------------------------------------------------------------------- the kernel
def _stem_dgrad_ref(dy7, dy3, w7, w3, H, W, absolute=False):
    """float64 autograd of the two stem convolutions (|dy|, |w| with ``absolute``: the bound's magnitude sum)."""
    f = (lambda t: t.abs()) if absolute else (lambda t: t)
    N = (dy7 if dy7 is not None else dy3).shape[0]
    x = torch.zeros(N, 3, H, W, dtype=torch.float64, requires_grad=True)
    loss = 0
    for dy, w, pad in ((dy7, w7, 3), (dy3, w3, 1)):
        if dy is not None:
            loss = loss + (F.conv2d(x, f(w.double()), None, 2, pad) * f(dy.double())).sum()
    (g,) = torch.autograd.grad(loss, x)
    return g


def _run_kernel(dt, dy7, dy3, w7, w3, H, W, ld_extra):
    """-> dx [N][3][H][W] from cabinet_stem_dgrad, after checking the canary margins around it."""
    lib = _lib.load()
    N = (dy7 if dy7 is not None else dy3).shape[0]
    OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1

    def nhwc(dy, C):
        if dy is None:
            return None, 0
        ld = C + ld_extra
        buf = torch.zeros(N, OH, OW, ld, dtype=TORCH_DT[dt], device="cuda")
        buf[..., :C] = dy.permute(0, 2, 3, 1).to("cuda", TORCH_DT[dt])
        return buf, ld

    b7, ld7 = nhwc(dy7, 64)
    b3, ld3 = nhwc(dy3, 16)
    margin, n = 256, N * 3 * H * W
    buf = torch.full((n + 2 * margin,), float("nan"), device="cuda")
    canary = torch.arange(2 * margin, dtype=torch.float32, device="cuda") * 1.25 - 7.0
    buf[:margin], buf[margin + n:] = canary[:margin], canary[margin:]
    w7d, w3d = w7.float().cuda().contiguous(), w3.float().cuda().contiguous()
    check(lib.cabinet_stem_dgrad(b7.data_ptr() if b7 is not None else None, ld7, b3.data_ptr() if b3 is not None else None,
                                 ld3, dt, w7d.data_ptr(), w3d.data_ptr(), buf[margin:].data_ptr(), N, H, W, OH, OW, stream()),
          "stem_dgrad")
    torch.cuda.synchronize()
    assert torch.equal(buf[:margin], canary[:margin]) and torch.equal(buf[margin + n:], canary[margin:])
    return buf[margin:margin + n].view(N, 3, H, W).cpu()


# (2, 400, 300): two 128-column strips per image and more class rows than SMs, so a CTA takes several rows and its
# share of rows crosses from one strip into the next
SIZES = [(1, 1, 1), (1, 2, 2), (2, 1, 5), (3, 4, 3), (2, 9, 16), (1, 70, 100), (2, 97, 131), (3, 33, 64), (2, 400, 300)]


@pytest.mark.parametrize("which", ["both", "no7", "no3"])
@pytest.mark.parametrize("N,H,W", SIZES)
@pytest.mark.parametrize("dt", [F32, BF16, F16], ids=["fp32", "bf16", "fp16"])
def test_stem_dgrad_kernel(dt, N, H, W, which):
    OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    tdt = TORCH_DT[dt]
    dy7 = None if which == "no7" else gen(N, 64, OH, OW, seed=1).to(tdt).float()
    dy3 = None if which == "no3" else gen(N, 16, OH, OW, seed=2).to(tdt).float()
    w7 = (gen(64, 3, 7, 7, seed=3) * 0.1).to(tdt).float()   # the kernel rounds the fp32 filters to the operand type
    w3 = (gen(16, 3, 3, 3, seed=4) * 0.3).to(tdt).float()
    ld_extra = 8 if (H + W) % 2 else 0
    dx = _run_kernel(dt, dy7, dy3, w7, w3, H, W, ld_extra)
    ref = _stem_dgrad_ref(dy7, dy3, w7, w3, H, W)
    mag = _stem_dgrad_ref(dy7, dy3, w7, w3, H, W, absolute=True)
    ulp = torch.from_numpy(np.spacing(np.abs(ref.numpy().astype(np.float32)))).double()
    err = (dx.double() - ref).abs()
    bound = 2.0 ** -16 * mag + ulp
    assert bool(torch.isfinite(dx).all())
    assert bool((err <= bound).all()), float((err - bound).max())
    assert torch.equal(dx, _run_kernel(dt, dy7, dy3, w7, w3, H, W, ld_extra))


# ----------------------------------------------------------------------------- the step, oracle helpers
def _sd(mode, C):
    return {k: v.clone() for k, v in build_model(C, mode).state_dict().items()}


def _ohem(N, H, W):
    thresh, n_min = 0.7, N * H * W // 16
    return lambda out, out16, lb: ohem_ce_loss(out, lb, thresh, n_min, 255) + ohem_ce_loss(out16, lb, thresh, n_min, 255)


def _smooth(C, N, H, W, aux_only=False):
    R = gen(N, C, H, W, seed=11) * 1e-3
    return lambda out, out16, lb: (out16 * R.to(out16)).sum() if aux_only else ((out + out16) * R.to(out)).sum()


def oracle_x_grad(sd, x, mode, loss_fn, lb, train, device="cpu", autocast=None, scale=1.0):
    """x.grad of the oracle network (train: batch statistics; eval: running statistics) under plain autograd."""
    sd = {k: v.to(device) for k, v in sd.items()}
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()
              if v.is_floating_point() and not k.endswith(("running_mean", "running_var"))}
    work = dict(sd)
    work.update(params)
    xg = x.to(device).float().clone().requires_grad_(True)
    cabinet_oracle.BATCH_STATS = {} if train else None
    try:
        with torch.autocast("cuda", dtype=autocast, enabled=autocast is not None):
            out, out16 = cabinet_oracle.cabinet_forward_graph(work, xg, BACKBONE_CFGS[mode])
            loss = loss_fn(out.float(), out16.float(), lb.to(device))
    finally:
        cabinet_oracle.BATCH_STATS = None
    (loss * scale).backward()
    return (xg.grad / scale).float().cpu()


def model_x_grad(model, x, loss_fn, lb, scale=1.0):
    xg = x.detach().clone().requires_grad_(True)
    out, out16 = model(xg)
    loss = loss_fn(out, out16, lb)
    (loss * scale).backward()
    return (xg.grad / scale).float().cpu(), out.detach(), loss.detach()


def _frozen_eval(model):
    model.eval()
    for p in model.parameters():
        p.requires_grad_(False)
    return model


# ----------------------------------------------------------------------------- nothing else changes
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_input_grad_changes_nothing_else(precision):
    mode, C, N, H, W = "large", 6, 2, 96, 80
    x, lb = make_input(N, H, W).cuda(), make_labels(N, H, W, C).cuda()
    crit = OhemCELoss(0.7, N * H * W // 16, 255)
    runs = []
    for need in (False, True, False, True):
        model = build_model(C, mode).cuda().train()
        model.train_precision = precision
        xi = x.clone().requires_grad_(need)
        out, out16 = model(xi)
        loss = crit(out, lb) + crit(out16, lb)
        loss.backward()
        assert (xi.grad is not None) == need
        runs.append((out.detach(), out16.detach(), loss.detach(),
                     {k: p.grad for k, p in model.named_parameters() if p.grad is not None},
                     {k: v for k, v in model.state_dict().items()}))
    for a, b in ((runs[0], runs[1]), (runs[2], runs[3])):
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
        assert a[3].keys() == b[3].keys() and all(torch.equal(a[3][k], b[3][k]) for k in a[3])
        assert all(torch.equal(a[4][k], b[4][k]) for k in a[4])


# ----------------------------------------------------------------------------- against the oracle
@pytest.mark.parametrize("loss_kind", ["ohem", "smooth"])
def test_train_mode_fp32_vs_oracle(loss_kind):
    mode, C, N, H, W = "large", 6, 2, 96, 80
    x, lb = make_input(N, H, W), make_labels(N, H, W, C)
    loss_fn = _ohem(N, H, W) if loss_kind == "ohem" else _smooth(C, N, H, W)
    ref = oracle_x_grad(_sd(mode, C), x, mode, loss_fn, lb, train=True)
    model = build_model(C, mode).cuda().train()
    model.train_precision = "fp32"
    got, _, _ = model_x_grad(model, x.cuda(), loss_fn, lb.cuda())
    e = rel_l2(got, ref)
    print(f"train fp32 {loss_kind}: x.grad rel_l2 {e:.3e}")
    assert e < 3e-2   # the whole step's parameter-gradient bar (test_gpu_train.py)


@pytest.mark.parametrize("aux_only", [False, True], ids=["both_outputs", "aux_only"])
def test_eval_mode_fp32_frozen_vs_oracle(aux_only):
    mode, C, N, H, W = "large", 6, 2, 96, 80
    x, lb = make_input(N, H, W), make_labels(N, H, W, C)
    loss_fn = _smooth(C, N, H, W, aux_only) if aux_only else _ohem(N, H, W)
    ref = oracle_x_grad(_sd(mode, C), x, mode, loss_fn, lb, train=False)
    model = _frozen_eval(build_model(C, mode).cuda())
    model.train_precision, model.precision = "fp32", "fp32"
    buffers = {k: v.clone() for k, v in model.named_buffers()}
    got, logits, _ = model_x_grad(model, x.cuda(), loss_fn, lb.cuda())
    e = rel_l2(got, ref)
    print(f"eval fp32 frozen ({'aux only' if aux_only else 'both outputs'}): x.grad rel_l2 {e:.3e}")
    assert e < 1e-3
    with torch.no_grad():
        infer, _ = model(x.cuda())
    assert infer.grad_fn is None
    assert rel_l2(logits.cpu(), infer.cpu()) < 1e-4
    assert all(p.grad is None for p in model.parameters())
    assert all(torch.equal(v, buffers[k]) for k, v in model.named_buffers())


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
def test_half_precision_within_the_reference_autocast_noise(precision, train):
    mode, C, N, H, W = "large", 6, 2, 96, 80
    x, lb = make_input(N, H, W), make_labels(N, H, W, C)
    loss_fn = _ohem(N, H, W)
    scale = 2.0 ** 16 if precision == "fp16" else 1.0   # GradScaler's default initial scale
    sd = _sd(mode, C)
    ref = oracle_x_grad(sd, x, mode, loss_fn, lb, train)
    ac = oracle_x_grad(sd, x, mode, loss_fn, lb, train, "cuda",
                       torch.float16 if precision == "fp16" else torch.bfloat16, scale)
    model = build_model(C, mode).cuda()
    model = model.train() if train else _frozen_eval(model)
    model.train_precision = precision
    got, _, _ = model_x_grad(model, x.cuda(), loss_fn, lb.cuda(), scale)
    e, bar = rel_l2(got, ref), 1.25 * rel_l2(ac, ref) + 0.01
    print(f"{precision} {'train' if train else 'eval'}: x.grad rel_l2 {e:.3e}, bar {bar:.3e}")
    assert bool(torch.isfinite(got).all()) and e <= bar


# ----------------------------------------------------------------------------- composition
def test_upstream_module_and_input_layouts():
    mode, C, N, H, W = "large", 6, 2, 96, 80
    x, lb = make_input(N, H, W), make_labels(N, H, W, C)
    loss_fn = _smooth(C, N, H, W)
    pre = torch.nn.Conv2d(3, 3, 3, padding=1)
    torch.nn.init.normal_(pre.weight, std=0.2, generator=torch.Generator().manual_seed(5))
    pre_ref = torch.nn.Conv2d(3, 3, 3, padding=1)
    pre_ref.load_state_dict(pre.state_dict())
    # the oracle: the same upstream convolution in front of the eval-mode oracle network
    sd = _sd(mode, C)
    cabinet_oracle.BATCH_STATS = None
    out, out16 = cabinet_oracle.cabinet_forward_graph(sd, pre_ref(x), BACKBONE_CFGS[mode])
    loss_fn(out, out16, lb).backward()
    model = _frozen_eval(build_model(C, mode).cuda())
    model.train_precision = "fp32"
    pre = pre.cuda()
    out, out16 = model(pre(x.cuda()))
    loss_fn(out, out16, lb.cuda()).backward()
    for got, want in ((pre.weight.grad, pre_ref.weight.grad), (pre.bias.grad, pre_ref.bias.grad)):
        assert rel_l2(got.cpu(), want) < 1e-3, rel_l2(got.cpu(), want)
    # fp16 and channels_last inputs: a gradient of their own dtype and shape, equal to the fp32 contiguous one
    x16 = x.cuda().half()
    g32, _, _ = model_x_grad(model, x16.float(), loss_fn, lb.cuda())
    xh = x16.clone().requires_grad_(True)
    loss_fn(*model(xh), lb.cuda()).backward()
    assert xh.grad.dtype == torch.float16 and xh.grad.shape == x16.shape
    assert torch.equal(xh.grad.cpu(), g32.half())
    xc = x16.float().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    loss_fn(*model(xc), lb.cuda()).backward()
    assert xc.grad.dtype == torch.float32 and xc.grad.shape == xc.shape
    assert torch.equal(xc.grad.cpu(), g32)


# ----------------------------------------------------------------------------- graph replay
def _pgd(model, x, lb, steps, keep_at=None):
    """sign-gradient steps on x (eval-mode attack) -> (trajectory, gradient kept at ``keep_at``, its copy)."""
    crit = OhemCELoss(0.7, x.shape[0] * x.shape[2] * x.shape[3] // 16, 255)
    xa, traj, kept = x.clone(), [], None
    for i in range(steps):
        xa.requires_grad_(True)
        out, out16 = model(xa)
        (g,) = torch.autograd.grad(crit(out, lb) + crit(out16, lb), xa)
        if i == keep_at:
            kept = (g, g.clone())
        xa = (xa.detach() + 0.01 * g.sign()).clamp(-3, 3)
        traj.append(xa)
    return traj, kept


def test_pgd_graph_replay_bit_identical_to_eager():
    mode, C, N, H, W = "large", 6, 2, 96, 80
    x, lb = make_input(N, H, W).cuda(), make_labels(N, H, W, C).cuda()
    trajs = []
    for graphed in (False, True):
        model = _frozen_eval(build_model(C, mode).cuda())
        model.train_precision = "bf16"
        eng = model.train_engine()
        eng.use_graph = graphed
        traj, kept = _pgd(model, x, lb, 9, keep_at=3)
        assert torch.equal(kept[0], kept[1])   # the replays after iteration 3 left the kept gradient alone
        if graphed:
            assert any(st.fwd is not None for st in eng._gsteps.values())
        trajs.append(traj)
    assert all(torch.equal(a, b) for a, b in zip(*trajs))


def test_adversarial_training_graph_replay_bit_identical_to_eager():
    """Eval-mode attack steps (frozen parameters, x requires grad) alternating with train steps on the adversarial
    batch: both geometries stay captured (max_graphs = 2) and every step matches the eager schedule bit for bit."""
    mode, C, N, H, W = "large", 6, 2, 96, 80
    crit = OhemCELoss(0.7, N * H * W // 16, 255)
    results = []
    for graphed in (False, True):
        model = build_model(C, mode).cuda()
        model.train_precision = "bf16"
        eng = model.train_engine()
        eng.use_graph = graphed
        opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9)
        advs = []
        for step in range(5):
            x, lb = make_input(N, H, W, seed=step).cuda(), make_labels(N, H, W, C, seed=step).cuda()
            model.eval()
            for p in model.parameters():
                p.requires_grad_(False)
            traj, _ = _pgd(model, x, lb, 2)
            for p in model.parameters():
                p.requires_grad_(True)
            model.train()
            opt.zero_grad(set_to_none=True)
            out, out16 = model(traj[-1])
            (crit(out, lb) + crit(out16, lb)).backward()
            opt.step()
            advs.append(traj[-1])
        if graphed:
            assert eng.max_graphs == 2 and sum(st.fwd is not None for st in eng._gsteps.values()) == 2
        results.append((advs, [p.detach().clone() for p in model.parameters()], list(model.buffers())))
    (a_adv, a_p, a_b), (b_adv, b_p, b_b) = results
    assert all(torch.equal(u, v) for u, v in zip(a_adv, b_adv))
    assert all(torch.equal(u, v) for u, v in zip(a_p, b_p))
    assert all(torch.equal(u, v) for u, v in zip(a_b, b_b))

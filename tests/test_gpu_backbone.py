"""GPU: MobileNetV3 run on its own.

* ``cabinet_stem3_tc`` (the backbone-only tensor-core stem) against fp32 conv + BN + HardSwish: odd heights, a strided
  output, geometries where every persistent CTA walks many tiles, and the refusal of W % 4 != 0 (which the engine routes
  to ``conv2d_simt``);
* eval-mode forward against the reference-generated ``stage_mobile_feat`` of the golden models, both inference
  precisions, fp32 and bf16 input, and at W % 4 != 0 against the oracle;
* train-mode forward + backward against autograd of ``oracle.cabinet_oracle.mobilenet`` with batch statistics: output,
  x.grad, every parameter gradient and every updated running statistic, at every ``train_precision`` (bf16 / fp16 bars
  calibrated against the oracle under autocast);
* frozen parameters / eval-mode BatchNorm children, the differentiable eval-mode call, engine invalidation, and
  ``net.mobile(x)`` inside a CABiNet.
"""

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from cabinet_b200 import MobileNetV3, _lib  # noqa: E402
from cabinet_b200._lib import check  # noqa: E402
from cabinet_b200.constants import BACKBONE_CFGS  # noqa: E402
from cabinet_b200.synthetic import build_model, make_input, state_dict_digest  # noqa: E402
from oracle import cabinet_oracle  # noqa: E402
from oracle.make_golden import MODEL_CASES  # noqa: E402
from tests.gpu_util import rel_l2  # noqa: E402

TOL = {"fp32": 1e-4, "bf16": 1e-2}   # the stage checks of test_gpu_parity.py


def make_backbone(mode, C=5):
    """A standalone MobileNetV3 carrying the (perturbed) backbone weights of the seeded CABiNet."""
    net = build_model(C, mode)
    mob = MobileNetV3(BACKBONE_CFGS[mode], mode, num_classes=C)
    mob.load_state_dict(net.mobile.state_dict())
    return mob.eval()


def oracle_sd(mob):
    return {"m." + k: v.detach().cpu().float().clone() for k, v in mob.state_dict().items()}


def oracle_forward(sd, x, mode):
    return cabinet_oracle.mobilenet(sd, x, BACKBONE_CFGS[mode], p="m")


# ---------------------------------------------------------------------------------------------------- the kernel
def _stem_ref(mob, x):
    conv, bn = mob.features[0][0], mob.features[0][1]
    return F.hardswish(F.batch_norm(F.conv2d(x, conv.weight.float(), None, 2, 1), bn.running_mean, bn.running_var,
                                    bn.weight, bn.bias, False, 0.0, bn.eps))


@pytest.mark.parametrize("N,H,W,ld", [(2, 64, 96, 16), (1, 33, 52, 16), (3, 97, 36, 24), (4, 512, 512, 16),
                                      (16, 256, 256, 16), (1, 2, 4, 16)])
def test_stem3_tc_against_fp32_conv_bn_hswish(N, H, W, ld):
    lib = _lib.load()
    mob = make_backbone("large").cuda()
    eng = mob.engine()
    x = torch.randn(N, 3, H, W, generator=torch.Generator().manual_seed(H * W + N)).cuda()
    OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    y = torch.full((N, OH, OW, ld), 7.0, dtype=torch.bfloat16, device="cuda")
    check(lib.cabinet_stem3_tc(x.data_ptr(), N, H, W, eng.stem_tc3.data_ptr(), y.data_ptr(), ld, OH, OW,
                               torch.cuda.current_stream().cuda_stream))
    with torch.no_grad():
        ref = _stem_ref(mob, x)
    e = rel_l2(y[..., :16].permute(0, 3, 1, 2).float().cpu(), ref.cpu())
    tiles = N * -(-OH // 16) * -(-OW // 8)
    print(f"stem3_tc N={N} {H}x{W} ld={ld} ({tiles} tiles): rel_l2 {e:.2e}")
    assert e < 8e-3   # bf16 input, weights and output: one rounding each
    assert bool((y[..., 16:] == 7.0).all())   # nothing written past the 16 channels


def test_stem3_tc_refuses_what_the_engine_routes_elsewhere():
    lib = _lib.load()
    eng = make_backbone("small").cuda().engine()
    x = torch.zeros(1, 3, 32, 70, device="cuda")
    y = torch.empty(1, 16, 35, 16, dtype=torch.bfloat16, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    assert lib.cabinet_stem3_tc(x.data_ptr(), 1, 32, 70, eng.stem_tc3.data_ptr(), y.data_ptr(), 16, 16, 35, s) == 1
    assert "multiple of 4" in lib.cabinet_last_error().decode()
    assert lib.cabinet_stem3_tc(x.data_ptr(), 1, 32, 68, eng.stem_tc3.data_ptr(), y.data_ptr(), 12, 16, 34, s) == 1
    assert lib.cabinet_stem3_tc(x.data_ptr(), 1, 32, 68, eng.stem_tc3.data_ptr(), y.data_ptr(), 16, 15, 34, s) == 1


# ---------------------------------------------------------------------------------------------------- eval mode
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name,mode,C,shape", MODEL_CASES)
def test_eval_matches_golden_stage(golden_dir, name, mode, C, shape, precision):
    g = np.load(golden_dir / f"model_{name}.npz")
    net = build_model(C, mode)
    assert state_dict_digest(net.state_dict()) == str(g["digest"])
    mob = MobileNetV3(BACKBONE_CFGS[mode], mode, num_classes=C)
    mob.load_state_dict(net.mobile.state_dict())
    mob = mob.cuda().eval()
    mob.precision = precision
    x = make_input(*shape).cuda()
    ref = torch.from_numpy(g["stage_mobile_feat"])
    dtypes = [torch.float32, torch.bfloat16] if precision == "bf16" else [torch.float32, torch.float16]
    for dt in dtypes:
        y = mob(x.to(dt))
        assert y.dtype == dt and y.shape == ref.shape and y.grad_fn is None and y.is_contiguous()
        e = rel_l2(y.float().cpu(), ref)
        print(f"{name} {precision} {dt}: stage mobile_feat rel_l2 {e:.3e}")
        assert e < (TOL[precision] if dt == torch.float32 else 1e-2), (dt, e)
    assert torch.equal(mob(x), mob(x))   # deterministic


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("mode,shape", [("small", (2, 64, 70)), ("large", (1, 45, 38))])
def test_eval_at_widths_the_tensor_core_stem_does_not_take(mode, shape, precision):
    mob = make_backbone(mode)
    x = make_input(*shape)
    with torch.no_grad():
        ref = oracle_forward(oracle_sd(mob), x, mode)
    mob = mob.cuda()
    mob.precision = precision
    y = mob(x.cuda())
    e = rel_l2(y.cpu(), ref)
    print(f"{mode} {shape} {precision}: rel_l2 {e:.3e}")
    assert e < TOL[precision]


def test_empty_batch_and_engine_invalidation():
    mob = make_backbone("small").cuda()
    assert mob(torch.zeros(0, 3, 64, 64, device="cuda")).shape == (0, 576, 2, 2)
    x = make_input(1, 64, 64).cuda()
    y0 = mob(x)
    with torch.no_grad():
        mob.conv[1].weight.mul_(2.0)   # a weight change is picked up
    y1 = mob(x)
    with torch.no_grad():
        ref = oracle_forward(oracle_sd(mob), x.cpu(), "small")
    assert not torch.equal(y0, y1) and rel_l2(y1.cpu(), ref) < TOL["bf16"]
    mob.to(torch.device("cuda"), torch.float32)
    assert mob.__dict__["_engine"] is None
    assert torch.equal(mob(x), y1)


# ---------------------------------------------------------------------------------------------------- train mode
def _oracle_train(sd, x, w, mode):
    """-> (y, x.grad, {param key: grad}, {bn prefix: (running_mean, running_var)}) of the oracle in train mode."""
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()
              if not k.endswith(("running_mean", "running_var", "num_batches_tracked")) and ".classifier." not in k}
    work = dict(sd)
    work.update(params)
    xg = x.clone().requires_grad_(True)
    cabinet_oracle.BATCH_STATS = {}
    try:
        y = oracle_forward(work, xg, mode)
        stats = cabinet_oracle.BATCH_STATS
    finally:
        cabinet_oracle.BATCH_STATS = None
    (y * w).sum().backward()
    running = {p: ((1 - 0.1) * sd[p + ".running_mean"] + 0.1 * m, (1 - 0.1) * sd[p + ".running_var"] + 0.1 * v)
               for p, (m, v, _) in stats.items()}
    return y.detach(), xg.grad, {k[2:]: p.grad for k, p in params.items()}, running


def _oracle_autocast(sd, x, w, mode, dtype):
    """The oracle's own deviation under torch.autocast(dtype) on the GPU (the reference's mixed-precision recipe)."""
    sdg = {k: v.cuda() for k, v in sd.items()}
    with torch.autocast("cuda", dtype=dtype):
        y, dx, grads, running = _oracle_train(sdg, x.cuda(), w.cuda(), mode)
    return (y.float().cpu(), dx.float().cpu(), {k: g.float().cpu() for k, g in grads.items()},
            {p: (m.float().cpu(), v.float().cpu()) for p, (m, v) in running.items()})


@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("mode,shape", [("large", (2, 128, 128)), ("small", (2, 96, 160))])
def test_train_matches_oracle(mode, shape, precision):
    N, H, W = shape
    mob = make_backbone(mode)
    sd = oracle_sd(mob)
    x = make_input(N, H, W)
    with torch.no_grad():
        w = torch.randn(oracle_forward(sd, x, mode).shape, generator=torch.Generator().manual_seed(5))
    y_ref, dx_ref, g_ref, run_ref = _oracle_train(sd, x, w, mode)
    bn_keys = [p[2:] for p in run_ref]
    mob = mob.cuda().train()
    mob.train_precision = precision
    xg = x.cuda().requires_grad_(True)
    y = mob(xg)
    assert y.dtype == torch.float32 and y.grad_fn is not None and y.shape == y_ref.shape
    (y * w.cuda()).sum().backward()
    assert xg.grad.dtype == torch.float32
    got = {"y": (y.detach().cpu(), y_ref), "x.grad": (xg.grad.cpu(), dx_ref)}
    for k, p in mob.named_parameters():
        if k.startswith("classifier"):
            assert p.grad is None, k
        else:
            got[k] = (p.grad.cpu(), g_ref[k])
    msd = mob.state_dict()
    for p in bn_keys:
        got[p + ".running_mean"] = (msd[p + ".running_mean"].cpu(), run_ref["m." + p][0])
        got[p + ".running_var"] = (msd[p + ".running_var"].cpu(), run_ref["m." + p][1])
        assert int(msd[p + ".num_batches_tracked"]) == int(sd["m." + p + ".num_batches_tracked"]) + 1
    typical = float(torch.tensor([float(b.norm()) for b in g_ref.values()]).median())
    if precision == "fp32":   # test_gpu_train.py: fp32 reductions in another order than ATen's
        bars = {k: 2e-3 for k in got}
    else:   # within 1.25 x the oracle's own deviation under autocast + 0.01 (test_gpu_train_fp16.py)
        ya, dxa, ga, ra = _oracle_autocast(sd, x, w, mode, torch.float16 if precision == "fp16" else torch.bfloat16)
        ac = {"y": ya, "x.grad": dxa, **ga}
        for p in bn_keys:
            ac[p + ".running_mean"], ac[p + ".running_var"] = ra["m." + p]
        bars = {k: 1.25 * rel_l2(ac[k], got[k][1]) + 0.01 for k in got}
    for k, (a, b) in got.items():
        e = rel_l2(a, b)
        print(f"train {mode} {shape} {precision} {k}: rel_l2 {e:.2e} (bar {bars[k]:.2e})")
        # a parameter gradient whose absolute error is below a tenth (fp32: a thousandth) of the median gradient norm
        # passes on that (BatchNorm affine gradients of the deepest blocks nearly cancel; test_gpu_train_fp16.py)
        small = k in g_ref and float((a - b).norm()) < (1e-3 if precision == "fp32" else 1e-1) * typical
        assert e <= bars[k] or small, (k, e, bars[k])


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_train_input_gradient_keeps_the_input_dtype(precision):
    mob = make_backbone("small").cuda().train()
    mob.train_precision = precision
    dt = torch.bfloat16 if precision == "bf16" else torch.float16
    xg = make_input(2, 64, 64).cuda().to(dt).requires_grad_(True)
    y = mob(xg)
    assert y.dtype == dt
    y.float().square().mean().backward()
    assert xg.grad.dtype == dt and torch.isfinite(xg.grad.float()).all() and xg.grad.float().abs().sum() > 0


def test_frozen_parameters_and_eval_bn_children():
    mob = make_backbone("large").cuda().train()
    for p in mob.features[0].parameters():
        p.requires_grad_(False)
    mob.features[3].conv[4].weight.requires_grad_(False)
    frozen_bns = ["features.5.conv.1", "conv.1"]
    mob.features[5].conv[1].eval()
    mob.conv[1].eval()
    before = {k: v.clone() for k, v in mob.state_dict().items()}
    x = make_input(2, 128, 128).cuda()
    mob(x).square().mean().backward()
    for n, p in mob.named_parameters():
        assert (p.grad is None) == (not p.requires_grad or n.startswith("classifier")), n
    msd = mob.state_dict()
    for p in frozen_bns:
        for leaf in ("running_mean", "running_var", "num_batches_tracked"):
            assert torch.equal(msd[f"{p}.{leaf}"], before[f"{p}.{leaf}"]), p
    assert not torch.equal(msd["features.0.1.running_mean"], before["features.0.1.running_mean"])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_eval_mode_input_gradient(precision):
    mob = make_backbone("small")
    sd = oracle_sd(mob)
    x = make_input(2, 96, 128)
    xr = x.clone().requires_grad_(True)
    y_ref = oracle_forward(sd, xr, "small")
    w = torch.randn(y_ref.shape, generator=torch.Generator().manual_seed(5))
    (y_ref * w).sum().backward()
    mob = mob.cuda().eval()
    mob.train_precision = precision
    before = {k: v.clone() for k, v in mob.state_dict().items()}
    xg = x.cuda().requires_grad_(True)
    y = mob(xg)
    assert y.grad_fn is not None
    (y * w.cuda()).sum().backward()
    if precision == "fp32":
        bar_y = bar_x = 2e-3
    else:   # within 1.25 x the oracle's own deviation under autocast + 0.01 (test_gpu_input_grad.py)
        xa = x.cuda().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            ya = oracle_forward({k: v.cuda() for k, v in sd.items()}, xa, "small")
        (ya.float() * w.cuda()).sum().backward()
        bar_y = 1.25 * rel_l2(ya.detach().float().cpu(), y_ref.detach()) + 0.01
        bar_x = 1.25 * rel_l2(xa.grad.float().cpu(), xr.grad) + 0.01
    ey, ex = rel_l2(y.detach().cpu(), y_ref.detach()), rel_l2(xg.grad.cpu(), xr.grad)
    print(f"eval-mode input gradient {precision}: y {ey:.2e} (bar {bar_y:.2e}), x.grad {ex:.2e} (bar {bar_x:.2e})")
    assert ey < bar_y and ex < bar_x
    assert all(torch.equal(v, before[k]) for k, v in mob.state_dict().items())
    assert mob.conv[0].weight.grad is not None and mob.classifier[0].weight.grad is None
    with torch.no_grad():
        assert mob(xg).grad_fn is None


# ---------------------------------------------------------------------------------------------------- inside a CABiNet
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_backbone_inside_cabinet(golden_dir, precision):
    name, mode, C, shape = MODEL_CASES[2]
    g = np.load(golden_dir / f"model_{name}.npz")
    net = build_model(C, mode).cuda()
    net.mobile.precision = precision
    y = net.mobile(make_input(*shape).cuda())
    e = rel_l2(y.cpu(), torch.from_numpy(g["stage_mobile_feat"]))
    print(f"net.mobile {precision}: rel_l2 {e:.2e}")
    assert e < TOL[precision]
    assert net.__dict__["_engine"] is None   # the backbone ran on its own engine
    f, _ = net(make_input(*shape).cuda())   # CABiNet's own schedule is unchanged
    assert rel_l2(f.cpu(), torch.from_numpy(g["final"])) < 1e-2

"""GPU: SpatialBranch, AttentionBranch, FeatureFusionModule and CABiNetOutput run on their own.

* ``cabinet_stem7_tc`` (sb.conv1 alone on the tensor cores) against fp32 conv + BN + ReLU: odd heights, a pixel stride
  > 64 with nothing written past channel 64, geometries where every persistent CTA walks many tiles, a 1 x 2 x 4 image,
  and the refusal of W % 4 != 0 and of a bad pixel stride;
* eval mode against the reference's own stage outputs of the golden models, each module fed the previous golden stage,
  both inference precisions and fp32 / bf16 / fp16 inputs, deterministic repeats;
* eval mode at widths CABiNet does not use, against the oracle (the spatial branch at W % 4 != 0: conv2d_simt);
* train mode against autograd of the oracle with batch statistics: outputs, every input gradient, every parameter
  gradient, every updated running statistic and ``num_batches_tracked``, at every ``train_precision``;
* AttentionBranch with only ``low`` or only ``high`` used; frozen parameters, eval-mode BN children, the differentiable
  eval-mode call, engine invalidation; two calls of one module before one backward, also under activation checkpointing;
* the modules of a CABiNet composed by hand reproduce ``net(x)``.
"""

import numpy as np
import pytest
import torch
import torch.nn.functional as F
import torch.utils.checkpoint

pytestmark = pytest.mark.gpu

from cabinet_b200 import AttentionBranch, CABiNetOutput, FeatureFusionModule, SpatialBranch, _lib  # noqa: E402
from cabinet_b200._lib import check  # noqa: E402
from cabinet_b200.synthetic import build_model, make_input, perturb_state_dict, state_dict_digest  # noqa: E402
from oracle import cabinet_oracle  # noqa: E402
from oracle.make_golden import MODEL_CASES  # noqa: E402
from tests.gpu_util import rel_l2  # noqa: E402

TOL = {"fp32": 1e-4, "bf16": 1e-2}   # the stage checks of test_gpu_parity.py

ORACLE = {   # module kind -> the oracle function of its forward, on a state_dict with the prefix "m."
    "sb": lambda sd, xs: (cabinet_oracle.spatial_branch(sd, xs[0], p="m"),),
    "ab": lambda sd, xs: tuple(cabinet_oracle.attention_branch(sd, xs[0], p="m")),
    "ffm": lambda sd, xs: (cabinet_oracle.ffm(sd, xs[0], xs[1], p="m"),),
    "head": lambda sd, xs: (cabinet_oracle.head(sd, xs[0], p="m"),),
}
CHILD = {"sb": "sb", "ab": "ab", "ffm": "ffm", "head": "conv_out"}


def oracle_sd(m):
    return {"m." + k: v.detach().cpu().float().clone() for k, v in m.state_dict().items()}


def perturbed(m, seed=3):
    m.load_state_dict(perturb_state_dict(m.state_dict(), seed))
    return m.eval()


def randn(*shape, seed=0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def as_tuple(y):
    return y if isinstance(y, tuple) else (y,)


# ---------------------------------------------------------------------------------------------------- the kernel
def _sb1_ref(sb, x):
    conv, bn = sb.conv1.conv, sb.conv1.bn
    return F.relu(F.batch_norm(F.conv2d(x, conv.weight.float(), None, 2, 3), bn.running_mean, bn.running_var, bn.weight,
                               bn.bias, False, 0.0, bn.eps))


@pytest.mark.parametrize("N,H,W,ld", [(2, 64, 96, 64), (1, 33, 52, 64), (3, 97, 36, 80), (4, 512, 512, 64),
                                      (16, 256, 256, 72), (1, 2, 4, 64)])
def test_stem7_tc_against_fp32_conv_bn_relu(N, H, W, ld):
    lib = _lib.load()
    sb = build_model(5, "large").sb.cuda()
    eng = sb.engine()
    x = randn(N, 3, H, W, seed=H * W + N).cuda()
    OH, OW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    y = torch.full((N, OH, OW, ld), 7.0, dtype=torch.bfloat16, device="cuda")
    check(lib.cabinet_stem7_tc(x.data_ptr(), N, H, W, eng.stem_tc7.data_ptr(), y.data_ptr(), ld, OH, OW,
                               torch.cuda.current_stream().cuda_stream))
    with torch.no_grad():
        ref = _sb1_ref(sb, x)
    e = rel_l2(y[..., :64].permute(0, 3, 1, 2).float().cpu(), ref.cpu())
    tiles = N * -(-OH // 16) * -(-OW // 8)
    print(f"stem7_tc N={N} {H}x{W} ld={ld} ({tiles} tiles): rel_l2 {e:.2e}")
    assert e < 8e-3   # bf16 input, weights and output: one rounding each
    assert bool((y[..., 64:] == 7.0).all())   # nothing written past the 64 channels


def test_stem7_tc_refuses_what_the_engine_routes_elsewhere():
    lib = _lib.load()
    eng = build_model(5, "small").sb.cuda().engine()
    x = torch.zeros(1, 3, 32, 70, device="cuda")
    y = torch.empty(1, 16, 35, 80, dtype=torch.bfloat16, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    w = eng.stem_tc7.data_ptr()
    assert lib.cabinet_stem7_tc(x.data_ptr(), 1, 32, 70, w, y.data_ptr(), 64, 16, 35, s) == 1
    assert "multiple of 4" in lib.cabinet_last_error().decode()
    for ld in (56, 68):   # below 64 channels, not a multiple of 8
        assert lib.cabinet_stem7_tc(x.data_ptr(), 1, 32, 68, w, y.data_ptr(), ld, 16, 34, s) == 1
        assert "ld_y" in lib.cabinet_last_error().decode()
    assert lib.cabinet_stem7_tc(x.data_ptr(), 1, 32, 68, w, y.data_ptr(), 64, 15, 34, s) == 1


# ---------------------------------------------------------------------------------------------------- eval mode
def _golden_inputs(g, kind):
    st = {k: torch.from_numpy(g["stage_" + k]) for k in ("feat_sb", "mobile_feat", "low", "feat_fuse")}
    if kind == "ffm":
        return [st["feat_sb"], cabinet_oracle.up(st["low"], st["feat_sb"].shape[2:])]
    return {"ab": [st["mobile_feat"]], "head": [st["feat_fuse"]]}[kind]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["sb", "ab", "ffm", "head"])
@pytest.mark.parametrize("name,mode,C,shape", MODEL_CASES)
def test_eval_matches_golden_stages(golden_dir, name, mode, C, shape, kind, precision):
    g = np.load(golden_dir / f"model_{name}.npz")
    net = build_model(C, mode)
    assert state_dict_digest(net.state_dict()) == str(g["digest"])
    m = getattr(net, CHILD[kind]).cuda().eval()
    m.precision = precision
    xs = [make_input(*shape)] if kind == "sb" else _golden_inputs(g, kind)
    refs = {"sb": ["feat_sb"], "ab": ["low", "high"], "ffm": ["feat_fuse"], "head": ["final8"]}[kind]
    dtypes = [torch.float32, torch.bfloat16, torch.float16]
    for dt in dtypes:
        ys = as_tuple(m(*[x.cuda().to(dt) for x in xs]))
        assert len(ys) == len(refs)
        for y, r in zip(ys, refs):
            ref = torch.from_numpy(g["stage_" + r])
            assert y.dtype == dt and y.shape == ref.shape and y.grad_fn is None and y.is_contiguous()
            e = rel_l2(y.float().cpu(), ref)
            print(f"{name} {kind} {precision} {dt}: stage {r} rel_l2 {e:.3e}")
            assert e < (TOL[precision] if dt == torch.float32 else 1e-2), (r, dt, e)
    xd = [x.cuda() for x in xs]
    assert all(torch.equal(a, b) for a, b in zip(as_tuple(m(*xd)), as_tuple(m(*xd))))   # deterministic


def _other_width(kind):
    """A module at widths CABiNet does not use, and its inputs."""
    torch.manual_seed(1)
    if kind == "sb":
        return perturbed(SpatialBranch()), [make_input(2, 64, 70)]   # W % 4 != 0: sb.conv1 on conv2d_simt
    if kind == "ab":
        return perturbed(AttentionBranch(512, 128, 128, 19)), [randn(2, 512, 16, 12, seed=2)]
    if kind == "ffm":
        return perturbed(FeatureFusionModule(64 + 128, 128)), [randn(2, 64, 24, 40, seed=3).relu(),
                                                               randn(2, 128, 24, 40, seed=4)]
    return perturbed(CABiNetOutput(128, 64, 19)), [randn(2, 128, 20, 36, seed=5).relu()]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["sb", "ab", "ffm", "head"])
def test_eval_at_other_widths_against_the_oracle(kind, precision):
    m, xs = _other_width(kind)
    with torch.no_grad():
        refs = ORACLE[kind](oracle_sd(m), xs)
    m = m.cuda()
    m.precision = precision
    ys = as_tuple(m(*[x.cuda() for x in xs]))
    for y, ref in zip(ys, refs):
        e = rel_l2(y.cpu(), ref)
        print(f"{kind} {tuple(ref.shape)} {precision}: rel_l2 {e:.3e}")
        assert y.shape == ref.shape and e < TOL[precision]


@pytest.mark.parametrize("kind", ["sb", "ab", "ffm", "head"])
def test_empty_batch_and_engine_invalidation(kind):
    m, xs = _other_width(kind)
    m = m.cuda()
    ys = as_tuple(m(*[torch.zeros((0,) + tuple(x.shape[1:]), device="cuda") for x in xs]))
    assert all(y.shape[0] == 0 for y in ys)
    xd = [x.cuda() for x in xs]
    y0 = as_tuple(m(*xd))
    with torch.no_grad():
        next(p for n, p in m.named_parameters() if n.endswith("bn.weight") or n.endswith("b2.weight")).mul_(2.0)
    y1 = as_tuple(m(*xd))
    with torch.no_grad():
        refs = ORACLE[kind](oracle_sd(m), xs)
    assert not all(torch.equal(a, b) for a, b in zip(y0, y1))
    assert all(rel_l2(a.cpu(), b) < TOL["bf16"] for a, b in zip(y1, refs))
    m.to(torch.device("cuda"), torch.float32)
    assert m.__dict__["_engine"] is None
    assert all(torch.equal(a, b) for a, b in zip(as_tuple(m(*xd)), y1))


# ---------------------------------------------------------------------------------------------------- train mode
def _oracle_train(kind, sd, xs, ws, train=True):
    """-> (outputs, input grads, {param key: grad}, {bn prefix: (running_mean, running_var)}) of the oracle's autograd."""
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()
              if not k.endswith(("running_mean", "running_var", "num_batches_tracked"))}
    work = dict(sd)
    work.update(params)
    xg = [x.clone().requires_grad_(True) for x in xs]
    cabinet_oracle.BATCH_STATS = {} if train else None
    try:
        ys = ORACLE[kind](work, xg)
        stats = cabinet_oracle.BATCH_STATS or {}
    finally:
        cabinet_oracle.BATCH_STATS = None
    sum((y.float() * w).sum() for y, w in zip(ys, ws) if w is not None).backward()
    running = {p: ((1 - 0.1) * sd[p + ".running_mean"] + 0.1 * mm, (1 - 0.1) * sd[p + ".running_var"] + 0.1 * v)
               for p, (mm, v, _) in stats.items()}
    return ([y.detach() for y in ys], [x.grad for x in xg], {k[2:]: p.grad for k, p in params.items()}, running)


def _oracle_autocast(kind, sd, xs, ws, dtype, train=True):
    sdg = {k: v.cuda() for k, v in sd.items()}
    with torch.autocast("cuda", dtype=dtype):
        ys, dxs, grads, running = _oracle_train(kind, sdg, [x.cuda() for x in xs],
                                                [w.cuda() if w is not None else None for w in ws], train)
    cpu = lambda t: t.float().cpu() if t is not None else None  # noqa: E731
    return ([cpu(y) for y in ys], [cpu(d) for d in dxs], {k: cpu(g) for k, g in grads.items()},
            {p: (cpu(a), cpu(b)) for p, (a, b) in running.items()})


def _train_case(kind):
    """A CABiNet-width module of the seeded model, and train-sized inputs."""
    net = build_model(5, "large")
    xs = {"sb": [make_input(2, 64, 96)], "ab": [randn(2, 960, 8, 16, seed=2).relu()],
          "ffm": [randn(2, 128, 16, 16, seed=3).relu(), randn(2, 256, 16, 16, seed=4)],
          "head": [randn(2, 256, 16, 16, seed=5).relu()]}[kind]
    return getattr(net, CHILD[kind]), xs


def _compare(got, ref, ac, precision, pgrad_keys, what):
    typical = float(torch.tensor([float(ref[k].norm()) for k in pgrad_keys]).median()) if pgrad_keys else 0.0
    for k, a in got.items():
        b = ref[k]
        bar = 2e-3 if precision == "fp32" else 1.25 * rel_l2(ac[k], b) + 0.01
        e = rel_l2(a, b)
        print(f"{what} {k}: rel_l2 {e:.2e} (bar {bar:.2e})")
        # a parameter gradient whose absolute error is below a tenth (fp32: a thousandth) of the median gradient norm
        # passes on that (test_gpu_backbone.py)
        small = k in pgrad_keys and float((a - b).norm()) < (1e-3 if precision == "fp32" else 1e-1) * typical
        assert e <= bar or small, (k, e, bar)


@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("kind", ["sb", "ab", "ffm", "head"])
def test_train_matches_oracle(kind, precision):
    m, xs = _train_case(kind)
    sd = oracle_sd(m)
    with torch.no_grad():
        ws = [randn(*y.shape, seed=9 + i) for i, y in enumerate(ORACLE[kind](sd, xs))]
    ys_ref, dx_ref, g_ref, run_ref = _oracle_train(kind, sd, xs, ws)
    m = m.cuda().train()
    m.train_precision = precision
    xg = [x.cuda().requires_grad_(True) for x in xs]
    ys = as_tuple(m(*xg))
    assert all(y.dtype == torch.float32 and y.grad_fn is not None for y in ys)
    sum((y * w.cuda()).sum() for y, w in zip(ys, ws)).backward()
    got = {f"y{i}": y.detach().cpu() for i, y in enumerate(ys)}
    ref = {f"y{i}": y for i, y in enumerate(ys_ref)}
    for i, x in enumerate(xg):
        assert x.grad.dtype == torch.float32
        got[f"x{i}.grad"], ref[f"x{i}.grad"] = x.grad.cpu(), dx_ref[i]
    for k, p in m.named_parameters():
        got[k], ref[k] = p.grad.cpu(), g_ref[k]
    msd = m.state_dict()
    for p, (rm, rv) in run_ref.items():
        k = p[2:]
        got[k + ".running_mean"], ref[k + ".running_mean"] = msd[k + ".running_mean"].cpu(), rm
        got[k + ".running_var"], ref[k + ".running_var"] = msd[k + ".running_var"].cpu(), rv
        assert int(msd[k + ".num_batches_tracked"]) == int(sd[p + ".num_batches_tracked"]) + 1
    assert len(run_ref) == sum(1 for mm in m.modules() if isinstance(mm, torch.nn.BatchNorm2d))
    ac = None
    if precision != "fp32":   # within 1.25 x the oracle's own deviation under autocast + 0.01 (test_gpu_train_fp16.py)
        ya, dxa, ga, ra = _oracle_autocast(kind, sd, xs, ws, torch.float16 if precision == "fp16" else torch.bfloat16)
        ac = {**{f"y{i}": y for i, y in enumerate(ya)}, **{f"x{i}.grad": d for i, d in enumerate(dxa)}, **ga}
        for p, (a, b) in ra.items():
            ac[p[2:] + ".running_mean"], ac[p[2:] + ".running_var"] = a, b
    _compare(got, ref, ac, precision, set(g_ref), f"train {kind} {precision}")


@pytest.mark.parametrize("kind", ["ab", "ffm", "head"])
def test_train_input_gradient_keeps_the_input_dtype(kind):
    m, xs = _train_case(kind)
    m = m.cuda().train()
    m.train_precision = "bf16"
    xg = [x.cuda().half().requires_grad_(True) for x in xs]
    ys = as_tuple(m(*xg))
    assert all(y.dtype == torch.float16 for y in ys)
    sum(y.float().square().mean() for y in ys).backward()
    for x in xg:
        assert x.grad.dtype == torch.float16 and torch.isfinite(x.grad.float()).all() and x.grad.float().abs().sum() > 0


@pytest.mark.parametrize("used", ["low", "high"])
def test_attention_branch_with_one_output_used(used):
    m, xs = _train_case("ab")
    sd = oracle_sd(m)
    with torch.no_grad():
        low, high = ORACLE["ab"](sd, xs)
    ws = [randn(*low.shape, seed=9), None] if used == "low" else [None, randn(*high.shape, seed=10)]
    ys_ref, dx_ref, g_ref, _ = _oracle_train("ab", sd, xs, ws)
    m = m.cuda().train()
    xg = xs[0].cuda().requires_grad_(True)
    lo, hi = m(xg)
    ((lo if used == "low" else hi) * (ws[0] if used == "low" else ws[1]).cuda()).sum().backward()
    unused = ("b1.", "b2.", "b4.") if used == "low" else ("convb.",)
    for k, p in m.named_parameters():
        if k.startswith(unused):
            assert p.grad is None and g_ref[k] is None, k
        else:
            e = rel_l2(p.grad.cpu(), g_ref[k])
            assert e < 2e-3 or float((p.grad.cpu() - g_ref[k]).norm()) < 1e-3 * float(g_ref[k].norm() + 1e-30), (k, e)
    e = rel_l2(xg.grad.cpu(), dx_ref[0])
    print(f"ab, only {used} used: x.grad rel_l2 {e:.2e}")
    assert e < 2e-3


def test_frozen_parameters_and_eval_bn_children():
    m, xs = _train_case("ab")
    m = m.cuda().train()
    m.conva[0].weight.requires_grad_(False)
    m.a2block.local_attn.refine[1].block[0].weight.requires_grad_(False)
    frozen_bns = ["b2", "a2block.global_attn.to_key.1"]
    m.b2.eval()
    m.a2block.global_attn.to_key[1].eval()
    before = {k: v.clone() for k, v in m.state_dict().items()}
    low, high = m(xs[0].cuda())
    (low.square().mean() + high.square().mean()).backward()
    for n, p in m.named_parameters():
        assert (p.grad is None) == (not p.requires_grad), n
    msd = m.state_dict()
    for p in frozen_bns:
        for leaf in ("running_mean", "running_var", "num_batches_tracked"):
            assert torch.equal(msd[f"{p}.{leaf}"], before[f"{p}.{leaf}"]), p
    assert not torch.equal(msd["conva.1.running_mean"], before["conva.1.running_mean"])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["sb", "ab", "ffm", "head"])
def test_eval_mode_input_gradient(kind, precision):
    m, xs = _train_case(kind)
    sd = oracle_sd(m)
    with torch.no_grad():
        ws = [randn(*y.shape, seed=9 + i) for i, y in enumerate(ORACLE[kind](sd, xs))]
    ys_ref, dx_ref, g_ref, _ = _oracle_train(kind, sd, xs, ws, train=False)
    m = m.cuda().eval()
    m.train_precision = precision
    before = {k: v.clone() for k, v in m.state_dict().items()}
    xg = [x.cuda().requires_grad_(i == 0) for i, x in enumerate(xs)]   # FFM: only fsp requires grad
    ys = as_tuple(m(*xg))
    assert all(y.grad_fn is not None for y in ys)
    sum((y * w.cuda()).sum() for y, w in zip(ys, ws)).backward()
    got = {**{f"y{i}": y.detach().cpu() for i, y in enumerate(ys)}, "x0.grad": xg[0].grad.cpu()}
    ref = {**{f"y{i}": y for i, y in enumerate(ys_ref)}, "x0.grad": dx_ref[0]}
    ac = None
    if precision != "fp32":
        ya, dxa, _, _ = _oracle_autocast(kind, sd, xs, ws, torch.bfloat16, train=False)
        ac = {**{f"y{i}": y for i, y in enumerate(ya)}, "x0.grad": dxa[0]}
    _compare(got, ref, ac, precision, set(), f"eval-mode grad {kind} {precision}")
    assert all(x.grad is None for x in xg[1:])
    assert all(torch.equal(v, before[k]) for k, v in m.state_dict().items())
    assert all(p.grad is not None for p in m.parameters())
    with torch.no_grad():
        assert as_tuple(m(*xg))[0].grad_fn is None


@pytest.mark.parametrize("kind", ["sb", "ab"])
def test_two_calls_before_one_backward(kind):
    """Two inputs through one module into one loss, and the same under activation checkpointing: each call keeps its
    own tape, so both backward passes see their own activations."""
    m, xs = _train_case(kind)
    x2 = [x.flip(-1) * 0.5 for x in xs]
    sd = oracle_sd(m)
    with torch.no_grad():
        ws = [randn(*y.shape, seed=9 + i) for i, y in enumerate(ORACLE[kind](sd, xs))]
    _, dx1_ref, g1, _ = _oracle_train(kind, sd, xs, ws, train=False)
    _, dx2_ref, g2, _ = _oracle_train(kind, sd, x2, ws, train=False)
    m = m.cuda().eval()
    for checkpointed in (False, True):
        m.zero_grad(set_to_none=True)
        a, b = [x.cuda().requires_grad_(True) for x in xs], [x.cuda().requires_grad_(True) for x in x2]
        run = ((lambda *t: torch.utils.checkpoint.checkpoint(m, *t, use_reentrant=False)) if checkpointed else m)
        ya, yb = as_tuple(run(*a)), as_tuple(run(*b))
        sum((y * w.cuda()).sum() for y, w in zip(ya + yb, ws + ws)).backward()
        errs = {"x1.grad": rel_l2(a[0].grad.cpu(), dx1_ref[0]), "x2.grad": rel_l2(b[0].grad.cpu(), dx2_ref[0])}
        for k, p in m.named_parameters():
            errs[k] = rel_l2(p.grad.cpu(), g1[k] + g2[k])
        worst = max(errs, key=errs.get)
        print(f"{kind} two calls, checkpointed={checkpointed}: worst {worst} rel_l2 {errs[worst]:.2e}")
        assert errs[worst] < 2e-3, (worst, errs[worst])


# ---------------------------------------------------------------------------------------------------- inside a CABiNet
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name,mode,C,shape", MODEL_CASES)
def test_modules_compose_to_cabinet(name, mode, C, shape, precision):
    net = build_model(C, mode).cuda().eval()
    net.precision = precision
    for child in (net.sb, net.mobile, net.ab, net.ffm, net.conv_out):
        child.precision = precision
    x = make_input(*shape).cuda()
    H, W = x.shape[2:]
    feat_sb = net.sb(x)
    low, high = net.ab(net.mobile(x))
    up = cabinet_oracle.up
    fuse = net.ffm(feat_sb, up(low, feat_sb.shape[2:]))
    final = up(net.conv_out(fuse), (H, W))
    aux = up(up(high, feat_sb.shape[2:]), (H, W))
    f_ref, a_ref = net(x)
    ef, ea = rel_l2(final.cpu(), f_ref.cpu()), rel_l2(aux.cpu(), a_ref.cpu())
    print(f"{name} {precision}: composed vs net(x): final {ef:.2e}, aux {ea:.2e}")
    assert ef < TOL[precision] and ea < TOL[precision]
    assert all(c.__dict__["_engine"] is not None for c in (net.sb, net.ab, net.ffm, net.conv_out))

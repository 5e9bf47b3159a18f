"""GPU: ContextAggregationBlock run on its own, at CABiNet's width and at others.

* ``cabinet_attention_tc_dkdv`` for every built (key width, value width) against fp32 softmax(q k^T dk^-1/2) v on the
  bf16-rounded inputs (whole, ragged and single key blocks; strided rows), and bit-identical to
  ``cabinet_attention_tc`` at 128 / 128;
* eval-mode forward against ``oracle.cabinet_oracle.cab`` at (C, V) in {(256, 128), (512, 128), (128, 64)}, both inference
  precisions, output dtype = input dtype;
* train-mode forward + backward against plain autograd of the oracle with batch statistics: output, x.grad, every
  parameter gradient (gamma included) and the five updated running statistics, at every ``train_precision``;
* frozen parameters / an eval-mode BatchNorm child, the differentiable eval-mode call, and the block inside a CABiNet.

Weights: every convolution re-initialised as ``AttentionBranch.init_weight`` does (a fresh block's ``project_out`` is
zero), then the perturbation of ``synthetic.perturb_state_dict`` (gamma = 0.5, randomised BatchNorm statistics / affine).
"""

import pytest
import torch
from torch import nn

pytestmark = pytest.mark.gpu

from cabinet_b200 import _lib  # noqa: E402
from cabinet_b200._lib import check  # noqa: E402
from cabinet_b200.modules import ContextAggregationBlock  # noqa: E402
from cabinet_b200.synthetic import build_model, perturb_state_dict  # noqa: E402
from oracle import cabinet_oracle  # noqa: E402
from tests.gpu_util import rel_l2  # noqa: E402

WIDTHS = [(256, 128), (512, 128), (128, 64)]
SHAPES = [(2, 32, 64), (1, 17, 23), (3, 32, 32)]
BN_KEYS = ("global_attn.to_query.1", "global_attn.to_key.1", "local_attn.refine.0.block.1",
           "local_attn.refine.1.block.1", "local_attn.refine.2.block.1")
FP32_TOL = 2e-5
# bf16 inference schedule (bf16 activations, folded bf16 weights, bf16 probabilities) against the fp32 oracle: measured
# 1.7e-3 ... 2.4e-3 rel-L2 over the widths and shapes below on a B200
BF16_TOL = 5e-3


def make_block(C, V, seed=0):
    torch.manual_seed(seed)
    blk = ContextAggregationBlock(C, V)
    for m in blk.modules():
        if isinstance(m, nn.Conv2d):
            nn.init.kaiming_normal_(m.weight, a=1)
    blk.load_state_dict(perturb_state_dict(blk.state_dict()))
    return blk.eval()


def oracle_sd(blk):
    return {"b." + k: v.detach().cpu().float().clone() for k, v in blk.state_dict().items()}


def make_x(N, C, H, W, seed=3):
    return torch.randn(N, C, H, W, generator=torch.Generator().manual_seed(seed))


# ---------------------------------------------------------------------------------------------------- the kernel
@pytest.mark.parametrize("dk,dv", [(64, 64), (64, 128), (128, 64), (128, 128), (256, 64), (256, 128)])
@pytest.mark.parametrize("L", [2048, 391, 128])
def test_attention_tc_dkdv(dk, dv, L):
    lib = _lib.load()
    N, pad = 2, 16
    g = torch.Generator().manual_seed(dk + dv + L)
    bufs = [torch.randn(N, L, d + pad, generator=g).to("cuda", torch.bfloat16) for d in (dk, dk, dv)]
    q, k, v = bufs[0][..., :dk], bufs[1][..., :dk], bufs[2][..., :dv]
    ctx = torch.zeros(N, L, dv + pad, dtype=torch.bfloat16, device="cuda")
    vt = torch.empty(N, dv, -(-L // 8) * 8, dtype=torch.bfloat16, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    check(lib.cabinet_attention_tc_dkdv(q.data_ptr(), dk + pad, k.data_ptr(), dk + pad, v.data_ptr(), dv + pad,
                                        vt.data_ptr(), ctx.data_ptr(), dv + pad, N, L, dk, dv, dk ** -0.5, stream))
    ref = torch.softmax(q.float() @ k.float().transpose(1, 2) * dk ** -0.5, dim=-1) @ v.float()
    e = rel_l2(ctx[..., :dv].float().cpu(), ref.cpu())
    print(f"attention_tc dk={dk} dv={dv} L={L}: rel_l2 {e:.2e}")
    assert e < 6e-3
    assert torch.count_nonzero(ctx[..., dv:]) == 0   # nothing written past the value width
    if dk == dv == 128:
        ctx2 = torch.zeros_like(ctx)
        check(lib.cabinet_attention_tc(q.data_ptr(), dk + pad, k.data_ptr(), dk + pad, v.data_ptr(), dv + pad,
                                       vt.data_ptr(), ctx2.data_ptr(), dv + pad, N, L, 128, dk ** -0.5, stream))
        assert torch.equal(ctx, ctx2)


# ---------------------------------------------------------------------------------------------------- eval mode
@pytest.mark.parametrize("C,V", WIDTHS)
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("precision,dtype", [("fp32", torch.float32), ("bf16", torch.float32), ("bf16", torch.bfloat16),
                                             ("fp32", torch.float16)])
def test_eval_matches_oracle(C, V, shape, precision, dtype):
    N, H, W = shape
    blk = make_block(C, V)
    sd = oracle_sd(blk)
    x = make_x(N, C, H, W).to(dtype)
    with torch.no_grad():
        ref = cabinet_oracle.cab(sd, "b", x.float())
    blk = blk.cuda()
    blk.precision = precision
    y = blk(x.cuda())
    assert y.dtype == dtype and y.shape == x.shape and y.grad_fn is None
    e = rel_l2(y.float().cpu(), ref)
    print(f"eval CAB({C}, {V}) {shape} {precision} {dtype}: rel_l2 {e:.2e}")
    bar = BF16_TOL if precision == "bf16" else (FP32_TOL if dtype == torch.float32 else 1e-3)  # fp16: output rounding
    assert e < bar
    assert torch.equal(blk(x.cuda()), y)   # deterministic


def _oracle_train(sd, x, w):
    """-> (y, x.grad, {param key: grad}, {bn prefix: (running_mean, running_var)}) of the oracle in train mode."""
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()
              if not k.endswith(("running_mean", "running_var", "num_batches_tracked"))}
    work = dict(sd)
    work.update(params)
    xg = x.clone().requires_grad_(True)
    cabinet_oracle.BATCH_STATS = {}
    try:
        y = cabinet_oracle.cab(work, "b", xg)
        stats = cabinet_oracle.BATCH_STATS
    finally:
        cabinet_oracle.BATCH_STATS = None
    (y * w).sum().backward()
    running = {p: ((1 - 0.1) * sd[p + ".running_mean"] + 0.1 * m, (1 - 0.1) * sd[p + ".running_var"] + 0.1 * v)
               for p, (m, v, _) in stats.items()}
    return y.detach(), xg.grad, {k[2:]: p.grad for k, p in params.items()}, running


def _oracle_autocast(sd, x, w, dtype):
    """The oracle's own deviation under torch.autocast(dtype) on the GPU (the reference's mixed-precision recipe)."""
    sdg = {k: v.cuda() for k, v in sd.items()}
    with torch.autocast("cuda", dtype=dtype):
        y, dx, grads, running = _oracle_train(sdg, x.cuda(), w.cuda())
    return (y.float().cpu(), dx.float().cpu(), {k: g.float().cpu() for k, g in grads.items()},
            {p: (m.float().cpu(), v.float().cpu()) for p, (m, v) in running.items()})


# ---------------------------------------------------------------------------------------------------- train mode
@pytest.mark.parametrize("C,V", WIDTHS)
@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("shape", [(2, 32, 64), (1, 17, 23)])
def test_train_matches_oracle(C, V, precision, shape):
    N, H, W = shape
    blk = make_block(C, V)
    sd = oracle_sd(blk)
    x = make_x(N, C, H, W)
    w = make_x(N, C, H, W, seed=5)
    y_ref, dx_ref, g_ref, run_ref = _oracle_train(sd, x, w)
    blk = blk.cuda().train()
    blk.train_precision = precision
    xg = x.cuda().requires_grad_(True)
    y = blk(xg)
    assert y.dtype == torch.float32 and y.grad_fn is not None
    (y * w.cuda()).sum().backward()
    got = {"y": (y.detach().cpu(), y_ref), "x.grad": (xg.grad.cpu(), dx_ref)}
    got.update({k: (p.grad.cpu(), g_ref[k]) for k, p in blk.named_parameters()})
    msd = blk.state_dict()
    for p in BN_KEYS:
        got[p + ".running_mean"] = (msd[p + ".running_mean"].cpu(), run_ref["b." + p][0])
        got[p + ".running_var"] = (msd[p + ".running_var"].cpu(), run_ref["b." + p][1])
        assert int(msd[p + ".num_batches_tracked"]) == 1
    typical = float(torch.tensor([float(b.norm()) for b in g_ref.values()]).median())
    if precision == "fp32":
        bars = {k: 1e-4 for k in got}
    else:   # within 1.25 x the oracle's own deviation under autocast + 0.01 (test_gpu_train_fp16.py)
        ya, dxa, ga, ra = _oracle_autocast(sd, x, w, torch.float16 if precision == "fp16" else torch.bfloat16)
        ac = {"y": ya, "x.grad": dxa, **ga}
        for p in BN_KEYS:
            ac[p + ".running_mean"], ac[p + ".running_var"] = ra["b." + p]
        bars = {k: 1.25 * rel_l2(ac[k], got[k][1]) + 0.01 for k in got}
    for k, (a, b) in got.items():
        e = rel_l2(a, b)
        print(f"train CAB({C}, {V}) {shape} {precision} {k}: rel_l2 {e:.2e} (bar {bars[k]:.2e})")
        # as in test_gpu_train_fp16.py: a parameter gradient whose absolute error is below a tenth of the median gradient
        # norm (the BatchNorm affine gradients of the local branch nearly cancel) passes on that
        small = precision != "fp32" and k in g_ref and float((a - b).norm()) < 1e-1 * typical
        assert e <= bars[k] or small, (k, e, bars[k])


def test_frozen_parameters_and_eval_bn_child():
    blk = make_block(512, 128).cuda().train()
    blk.gamma.requires_grad_(False)
    blk.global_attn.to_key[0].weight.requires_grad_(False)
    blk.local_attn.refine[1].block[1].eval()
    before = {k: v.clone() for k, v in blk.state_dict().items()}
    x = make_x(2, 512, 32, 64).cuda()
    blk(x).square().mean().backward()
    for n, p in blk.named_parameters():
        assert (p.grad is None) == (not p.requires_grad), n
    msd = blk.state_dict()
    frozen = "local_attn.refine.1.block.1"
    for leaf in ("running_mean", "running_var", "num_batches_tracked"):
        assert torch.equal(msd[f"{frozen}.{leaf}"], before[f"{frozen}.{leaf}"])
    for p in BN_KEYS:
        if p != frozen:
            assert not torch.equal(msd[p + ".running_mean"], before[p + ".running_mean"]), p


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_eval_mode_input_gradient(precision):
    blk = make_block(256, 128)
    sd = oracle_sd(blk)
    x, w = make_x(2, 256, 32, 64), make_x(2, 256, 32, 64, seed=5)
    xr = x.clone().requires_grad_(True)
    y_ref = cabinet_oracle.cab(sd, "b", xr)
    (y_ref * w).sum().backward()
    blk = blk.cuda().eval()
    blk.train_precision = precision
    before = {k: v.clone() for k, v in blk.state_dict().items()}
    xg = x.cuda().requires_grad_(True)
    y = blk(xg)
    assert y.grad_fn is not None
    (y * w.cuda()).sum().backward()
    bar = 1e-4 if precision == "fp32" else 2e-2
    assert rel_l2(y.detach().cpu(), y_ref.detach()) < bar
    assert rel_l2(xg.grad.cpu(), xr.grad) < bar
    assert all(torch.equal(v, before[k]) for k, v in blk.state_dict().items())
    assert blk.gamma.grad is not None


@pytest.mark.parametrize("precision,bar", [("fp32", FP32_TOL), ("bf16", BF16_TOL)])
def test_block_inside_cabinet(precision, bar):
    net = build_model(5, "large").cuda()
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    feat = torch.relu(make_x(2, 256, 16, 16))
    with torch.no_grad():
        ref = cabinet_oracle.cab(sd, "ab.a2block", feat)
    net.ab.a2block.precision = precision
    y = net.ab.a2block(feat.cuda())
    e = rel_l2(y.cpu(), ref)
    print(f"net.ab.a2block {precision}: rel_l2 {e:.2e}")
    assert e < bar
    assert net.__dict__["_engine"] is None   # the block ran on its own engine

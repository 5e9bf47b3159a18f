"""ORACLE (test infrastructure, not product code) — CPU restatement of ``CABiNet.forward``.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this file.  The product path
(``cabinet_b200``) never does, and raises if its CUDA library is missing.

What this is: a functional, state_dict-driven restatement of the reference's forward
algorithm in fp32 on CPU.  The arithmetic primitives of the reference live in a
third-party dependency (PyTorch ATen, ``torch>=2.0.0`` unpinned in the reference's
``pyproject.toml:13``; 2.11.0+cu128 installed here), so the restatement is written
against the same primitives (``F.conv2d``, ``F.batch_norm`` maths, ``F.interpolate``,
``F.adaptive_avg_pool2d``, ``softmax``) with every function citing the reference
``file:line`` it follows.  ``oracle/primitives_np.py`` additionally restates the two
index-rule primitives (bilinear ``align_corners=False`` and adaptive-avg-pool bins) in
plain numpy, which is what the CUDA kernels implement.

Pinning: the reference's own tests hold no golden values for this path (SURVEY §8c), so the
oracle is pinned against outputs of the *imported, unmodified reference* generated in the
build container by ``oracle/make_golden.py`` and committed under ``tests/golden/``
(``tests/test_oracle_golden.py``).
"""

from __future__ import annotations

import torch
import torch.nn.functional as F

BN_EPS = 1e-5
PSP_SIZES = (1, 3, 6, 8)


# ----------------------------------------------------------------------------- primitives
def make_divisible(v, divisor=8, min_value=None):
    # reference: src/models/mobilenetv3.py:18-35
    if min_value is None:
        min_value = divisor
    new_v = max(min_value, int(v + divisor / 2) // divisor * divisor)
    if new_v < 0.9 * v:
        new_v += divisor
    return new_v


# Train-mode BatchNorm (oracle/train_oracle.py, the training step of BASELINE config 5): when this dict is not None,
# ``bn`` normalises with the statistics of the batch (nn.BatchNorm2d in .train(), src/models/cabinet.py:30-31 etc.) and
# records them so the caller can restate the running-statistics update.  None (the default) = inference.
BATCH_STATS = None


def bn(sd, prefix, x):
    """BatchNorm2d.  Eval mode: (x-mean)/sqrt(var+eps)*gamma+beta (ATen native_batch_norm, eval)."""
    if BATCH_STATS is not None:
        BATCH_STATS[prefix] = (x.detach().mean(dim=(0, 2, 3)), x.detach().var(dim=(0, 2, 3), unbiased=True),
                               x.shape[0] * x.shape[2] * x.shape[3])
        return F.batch_norm(x, None, None, sd[prefix + ".weight"], sd[prefix + ".bias"], True, 0.0, BN_EPS)
    return F.batch_norm(x, sd[prefix + ".running_mean"], sd[prefix + ".running_var"], sd[prefix + ".weight"],
                        sd[prefix + ".bias"], False, 0.0, BN_EPS)


def hard_sigmoid(x):
    return F.relu6(x + 3) / 6  # reference: mobilenetv3.py:38-50


def hard_swish(x):
    return x * hard_sigmoid(x)  # reference: mobilenetv3.py:53-65


def act(x, hs):
    return hard_swish(x) if hs else F.relu(x)


def up(x, size):
    return F.interpolate(x, size=size, mode="bilinear", align_corners=False)


# ----------------------------------------------------------------------------- backbone
def se_layer(sd, p, x):
    # reference: mobilenetv3.py:68-83 — GAP -> Linear -> ReLU -> Linear -> hard-sigmoid -> scale
    b, c = x.shape[:2]
    y = x.mean(dim=(2, 3))
    y = F.relu(F.linear(y, sd[p + ".fc.0.weight"], sd[p + ".fc.0.bias"]))
    y = hard_sigmoid(F.linear(y, sd[p + ".fc.2.weight"], sd[p + ".fc.2.bias"]))
    return x * y.view(b, c, 1, 1)


def inverted_residual(sd, p, x, blk):
    # reference: mobilenetv3.py:102-159 (ordering F10: SE sits before the activation in the expand form)
    k, s, hs, se = blk["k"], blk["s"], blk["hs"], blk["se"]
    pad = (k - 1) // 2
    c = p + ".conv"
    if not blk["expand"]:
        y = F.conv2d(x, sd[c + ".0.weight"], None, s, pad, 1, blk["exp"])
        y = act(bn(sd, c + ".1", y), hs)
        if se:
            y = se_layer(sd, c + ".3", y)
        y = bn(sd, c + ".5", F.conv2d(y, sd[c + ".4.weight"]))
    else:
        y = act(bn(sd, c + ".1", F.conv2d(x, sd[c + ".0.weight"])), hs)
        y = F.conv2d(y, sd[c + ".3.weight"], None, s, pad, 1, blk["exp"])
        y = bn(sd, c + ".4", y)
        if se:
            y = se_layer(sd, c + ".5", y)
        y = act(y, hs)
        y = bn(sd, c + ".8", F.conv2d(y, sd[c + ".7.weight"]))
    return x + y if blk["identity"] else y


def resolve_blocks(cfgs):
    # reference: mobilenetv3.py:172-185
    inp = make_divisible(16, 8)
    out, exp = [], inp
    for k, t, c, se, hs, s in cfgs:
        oc = make_divisible(c, 8)
        exp = make_divisible(inp * t, 8)
        out.append(dict(inp=inp, exp=exp, out=oc, k=int(k), s=int(s), se=bool(se), hs=bool(hs),
                        identity=(int(s) == 1 and inp == oc), expand=(inp != exp)))
        inp = oc
    return out


def mobilenet(sd, x, cfgs, p="mobile"):
    # reference: mobilenetv3.py:86-91,173,202-205 — stem 3x3 s2 + BN + HS, blocks, 1x1 + BN + HS
    y = hard_swish(bn(sd, p + ".features.0.1", F.conv2d(x, sd[p + ".features.0.0.weight"], None, 2, 1)))
    for i, blk in enumerate(resolve_blocks(cfgs)):
        y = inverted_residual(sd, f"{p}.features.{i + 1}", y, blk)
    return hard_swish(bn(sd, p + ".conv.1", F.conv2d(y, sd[p + ".conv.0.weight"])))


# ----------------------------------------------------------------------------- CAB
def psp(sd, p, x, sizes=PSP_SIZES):
    # reference: cab.py:65-76 — priors are pooled then upsampled BACK to (h, w) (F5), then 1x1 5C->C
    h, w = x.shape[2:]
    priors = [x] + [up(F.adaptive_avg_pool2d(x, (s, s)), (h, w)) for s in sizes]
    return F.conv2d(torch.cat(priors, dim=1), sd[p + ".project.weight"])


def global_attention(sd, p, x):
    # reference: cab.py:131-162 with scale == 1 (pool = Identity, no final interpolate)
    B, _, H, W = x.shape
    q = F.relu(bn(sd, p + ".to_query.1", F.conv2d(x, sd[p + ".to_query.0.weight"])))
    q = q.view(B, -1, H * W).transpose(1, 2)
    k = psp(sd, p + ".psp_key", F.relu(bn(sd, p + ".to_key.1", F.conv2d(x, sd[p + ".to_key.0.weight"]))))
    k = k.view(B, -1, H * W)
    v = psp(sd, p + ".psp_value", F.conv2d(x, sd[p + ".to_value.weight"]))
    v = v.view(B, -1, H * W).transpose(1, 2)
    attn = torch.bmm(q, k) * (k.shape[1] ** -0.5)
    attn = F.softmax(attn, dim=-1)
    ctx = torch.bmm(attn, v).transpose(1, 2).reshape(B, -1, H, W)
    return F.conv2d(ctx, sd[p + ".project_out.weight"])


def local_attention(sd, p, x):
    # reference: cab.py:18-38,170-184 — x + x * sigmoid(DW3(DW3(DW3(x)))), DW3 = dw3x3 + BN + ReLU
    r = x
    for i in range(3):
        b = f"{p}.refine.{i}.block"
        r = F.relu(bn(sd, b + ".1", F.conv2d(r, sd[b + ".0.weight"], None, 1, 1, 1, r.shape[1])))
    return x + x * torch.sigmoid(r)


def cab(sd, p, x):
    # reference: cab.py:213-216
    return sd[p + ".gamma"] * global_attention(sd, p + ".global_attn", x) + local_attention(sd, p + ".local_attn", x)


# ----------------------------------------------------------------------------- CABiNet
def conv_bn_relu(sd, p, x, stride, pad):
    # reference: cabinet.py:19-44
    return F.relu(bn(sd, p + ".bn", F.conv2d(x, sd[p + ".conv.weight"], None, stride, pad)))


def spatial_branch(sd, x, p="sb"):
    # reference: cabinet.py:108-129
    x = conv_bn_relu(sd, p + ".conv1", x, 2, 3)
    x = conv_bn_relu(sd, p + ".conv2", x, 2, 1)
    x = conv_bn_relu(sd, p + ".conv3", x, 2, 1)
    return conv_bn_relu(sd, p + ".conv_out", x, 1, 0)


def attention_branch(sd, x, p="ab"):
    # reference: cabinet.py:75-94
    feat = F.relu(bn(sd, p + ".conva.1", F.conv2d(x, sd[p + ".conva.0.weight"], None, 1, 1)))
    feat = cab(sd, p + ".a2block", feat)
    low = F.conv2d(feat, sd[p + ".convb.weight"], sd[p + ".convb.bias"])
    fused = F.conv2d(torch.cat([x, feat], dim=1), sd[p + ".b1.weight"], None, 1, 1)
    fused = F.relu(bn(sd, p + ".b2", fused))
    high = F.conv2d(fused, sd[p + ".b4.weight"], sd[p + ".b4.bias"])
    return low, high


def ffm(sd, fsp, fcp, p="ffm"):
    # reference: cabinet.py:142-153
    feat = conv_bn_relu(sd, p + ".convblk", torch.cat([fsp, fcp], dim=1), 1, 0)
    att = feat.mean(dim=(2, 3), keepdim=True)
    att = torch.sigmoid(F.conv2d(F.relu(F.conv2d(att, sd[p + ".conv1.weight"])), sd[p + ".conv2.weight"]))
    return feat * att + feat


def head(sd, x, p="conv_out"):
    # reference: cabinet.py:162-172
    return F.conv2d(conv_bn_relu(sd, p + ".conv", x, 1, 1), sd[p + ".conv_out.weight"])


@torch.no_grad()
def cabinet_forward(sd, x, cfgs, stages=None):
    """fp32 CPU forward of the whole path.  ``sd`` = state_dict (CPU fp32), ``x`` = (N,3,H,W) fp32.

    reference: cabinet.py:207-247.  If ``stages`` is a dict it receives the intermediate activations
    (NCHW fp32) under the names the parity tests use.
    """
    sd = {k: v.detach().to("cpu") for k, v in sd.items()}
    x = x.detach().to("cpu", torch.float32)
    return cabinet_forward_graph(sd, x, cfgs, stages)


def cabinet_forward_graph(sd, x, cfgs, stages=None):
    """The same forward without ``no_grad`` / detach: differentiable w.r.t. the tensors of ``sd`` (train oracle)."""
    H, W = x.shape[2:]
    feat_sb = spatial_branch(sd, x)
    mobile_feat = mobilenet(sd, x, cfgs)
    low, high = attention_branch(sd, mobile_feat)
    low_up = up(low, feat_sb.shape[2:])
    high_up = up(high, feat_sb.shape[2:])
    feat_fuse = ffm(sd, feat_sb, low_up)
    final8 = head(sd, feat_fuse)
    final = up(final8, (H, W))
    aux = up(high_up, (H, W))  # two-stage upsample of the aux head (F8)
    if stages is not None:
        stages.update(feat_sb=feat_sb, mobile_feat=mobile_feat, low=low, high=high, feat_fuse=feat_fuse,
                      final8=final8)
    return final, aux

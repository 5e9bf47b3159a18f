"""No GPU: the standalone MobileNetV3's validation, parameter surface, engine housekeeping, its inference and training
schedules against the recording double of the C-ABI, and the compiled backbone-only stem kernel."""

import copy
import pickle
import re
import shutil
import subprocess
from pathlib import Path

import pytest
import torch

from cabinet_b200 import MobileNetV3, _lib, engine as engine_mod
from cabinet_b200.constants import BACKBONE_CFGS
from cabinet_b200.modules import CABiNet
from tests.test_engine_dryrun import RecordingLib

BRANCH_PREFIXES = ("sb.", "ab.", "ffm.", "cab.", "conv_out.", "low_up", "high_up", "final_up", "aux_up")


def backbone(mode="large", **kw):
    return MobileNetV3(BACKBONE_CFGS[mode], mode, **kw)


class _P:  # parameters that claim to live on a CUDA device
    is_cuda = True
    device = torch.device("cpu")


# ---------------------------------------------------------------------------------------------------- validation
def test_cpu_input_raises():
    with pytest.raises(RuntimeError, match="no CPU path"):
        backbone()(torch.randn(1, 3, 32, 32))


@pytest.mark.parametrize("dtype", [torch.float64, torch.int32, torch.uint8])
def test_other_dtypes_raise(dtype):
    with pytest.raises(TypeError, match="float32, bfloat16 or float16"):
        backbone("small")(torch.zeros(1, 3, 32, 32, dtype=dtype))


@pytest.mark.parametrize("shape", [(1, 4, 32, 32), (1, 1, 32, 32), (3, 32, 32)])
def test_wrong_shape_raises(shape):
    with pytest.raises(ValueError, match=r"\(N, 3, H, W\)"):
        backbone()(torch.randn(*shape))


def test_width_mult_raises_at_the_first_call():
    net = backbone("small", width_mult=0.75)   # the parameter tree itself builds
    with pytest.raises(ValueError, match="width_mult"):
        net(torch.randn(1, 3, 32, 32))


# ---------------------------------------------------------------------------------------------------- module surface
@pytest.mark.parametrize("mode", ["large", "small"])
def test_state_dict_keys_equal_cabinets_backbone(mode):
    keys = list(backbone(mode).state_dict())
    net_keys = list(CABiNet(5, mode=mode).state_dict())
    assert keys == [k[len("mobile."):] for k in net_keys if k.startswith("mobile.")]
    assert all("precision" not in k and "engine" not in k for k in keys)


def test_exported_and_attributes_default_like_cabinet():
    import cabinet_b200

    assert "MobileNetV3" in cabinet_b200.__all__ and cabinet_b200.MobileNetV3 is MobileNetV3
    mob, net = backbone("small"), CABiNet(5, mode="small")
    assert (mob.precision, mob.train_precision) == (net.precision, net.train_precision) == ("bf16", "fp32")
    assert mob.out_channels == 576 and backbone().out_channels == 960


def _with_engines(m):
    m.__dict__["_engine"], m.__dict__["_train_engine"] = object(), object()
    return m


def test_deepcopy_and_pickle_carry_no_engine():
    mob = _with_engines(backbone("small"))
    for new in (copy.deepcopy(mob), pickle.loads(pickle.dumps(mob))):
        assert new.__dict__["_engine"] is None and new.__dict__["_train_engine"] is None
        assert new.state_dict().keys() == mob.state_dict().keys()
    assert mob.__dict__["_engine"] is not None   # the original keeps its engines
    net = _with_engines(CABiNet(5, mode="small"))
    _with_engines(net.mobile)
    new = copy.deepcopy(net)
    assert new.mobile.__dict__["_engine"] is None and new.mobile.__dict__["_train_engine"] is None


def test_apply_drops_engines():
    mob = _with_engines(backbone("small"))
    mob.float()
    assert mob.__dict__["_engine"] is None and mob.__dict__["_train_engine"] is None
    net = CABiNet(5, mode="small")
    _with_engines(net.mobile)
    net.float()   # the nested backbone's engines go too
    assert net.mobile.__dict__["_engine"] is None and net.mobile.__dict__["_train_engine"] is None


def test_weight_change_is_seen_by_the_stamp():
    mob = backbone("small")
    s0 = mob._weights_stamp()
    with torch.no_grad():
        mob.conv[0].weight.mul_(2)
    assert mob._weights_stamp() != s0


# ---------------------------------------------------------------------------------------------------- dry runs
def _record(monkeypatch, module, cls_module, cls, *args):
    rec = RecordingLib()
    rec.cabinet_train_scratch_floats = lambda M, C, nq: 16
    rec.cabinet_conv_wgrad_scratch_floats = lambda *a: 16
    rec.cabinet_conv_wgrad_tc_scratch_floats = lambda *a: 16
    monkeypatch.setattr(_lib, "load", lambda: rec)
    monkeypatch.setattr(cls, "stream", property(lambda self: None))
    real_next = next
    monkeypatch.setattr(cls_module, "next", lambda it: _P, raising=False)
    eng = cls(module, *args)
    monkeypatch.setattr(cls_module, "next", real_next, raising=False)
    return eng, rec


@pytest.mark.parametrize("mode,precision,W", [("large", "bf16", 96), ("small", "bf16", 64), ("large", "fp32", 64),
                                              ("small", "bf16", 70)])
def test_inference_schedule_is_the_backbone_alone(monkeypatch, mode, precision, W):
    mob = backbone(mode).eval()
    eng, rec = _record(monkeypatch, mob, engine_mod, engine_mod.Engine, precision)
    assert not hasattr(eng, "sb1") and not hasattr(eng, "to_q") and not hasattr(eng, "stem_tc2")
    layers = []
    run = eng._run
    monkeypatch.setattr(eng, "_run", lambda kernel, layer, *a: (layers.append(layer), run(kernel, layer, *a))[1])
    x = torch.zeros(2, 3, 64, W)
    y = eng.forward_backbone(x)
    assert y.shape == (2, mob.out_channels, 2, -(-W // 32)) and y.dtype == x.dtype
    names = [c[0] for c in rec.calls]
    tc_stem = precision == "bf16" and W % 4 == 0
    assert names.count("cabinet_stem3_tc") == (1 if tc_stem else 0)
    assert "cabinet_stem_tc2" not in names and "cabinet_stem_tc" not in names
    assert layers.count("mobile.stem") == 1 and layers[0] == "mobile.stem"
    assert (names[0] == "cabinet_stem3_tc") if tc_stem else (names[0] == "cabinet_conv2d_simt")
    assert not [n for n in layers if n.startswith(BRANCH_PREFIXES)], layers
    assert layers[-2:] == ["mobile.conv", "mobile.out"] and names[-1] == "cabinet_resample_sep"
    n_blocks = 15 if mode == "large" else 11
    assert (names.count("cabinet_dwconv") + names.count("cabinet_dwconv_tma") + names.count("cabinet_mbconv_noexpand_fused")
            + names.count("cabinet_mbconv_fused") + names.count("cabinet_mbconv_t")) == n_blocks
    extra = 1 + names.count("cabinet_channel_sum")   # the SE-sum memset (+ the fp32 mode's channel-sum scratch)
    assert eng.launches == len(names) + extra
    if tc_stem:
        a = dict(zip(("x", "N", "H", "W", "w", "y", "ld", "OH", "OW"), rec.calls[0][1]))
        assert (a["N"], a["H"], a["W"], a["ld"], a["OH"], a["OW"]) == (2, 64, W, 16, 32, W // 2)
        assert tuple(eng.stem_tc3.shape) == (3, 2, 16, 8) and eng.stem_tc3.dtype == torch.bfloat16


def test_inference_engine_refuses_packed_weights_for_a_backbone(monkeypatch):
    with pytest.raises(ValueError, match="CABiNet engines only"):
        _record(monkeypatch, backbone("small"), engine_mod, engine_mod.Engine, "bf16", {"stem": None})


def test_stem3_weights_hold_the_folded_filter_and_bias(monkeypatch):
    mob = backbone("small").eval()
    eng, _ = _record(monkeypatch, mob, engine_mod, engine_mod.Engine, "bf16")
    w3, b3 = engine_mod._fold(mob.features[0][0].weight, None, mob.features[0][1])
    wn = eng.stem_tc3.float().permute(2, 0, 1, 3).reshape(16, 3, 4, 4)   # [o][ky][slot][c]
    assert torch.allclose(wn[:, :, 1:, :3], w3.permute(0, 2, 3, 1).to(torch.bfloat16).float())
    assert torch.allclose(wn[:, 1, 0, 3] + wn[:, 0, 0, 3], b3, rtol=1e-4, atol=1e-6)
    assert torch.count_nonzero(wn[:, :, 0, :3]) == 0 and torch.count_nonzero(wn[:, 2, 0, 3]) == 0
    assert torch.count_nonzero(wn[:, :, 1:, 3]) == 0


@pytest.mark.parametrize("mode,precision", [("large", "bf16"), ("small", "bf16"), ("large", "fp32"), ("small", "fp16")])
@pytest.mark.parametrize("input_grad", [False, True])
def test_training_schedule_is_the_backbone_alone(monkeypatch, mode, precision, input_grad):
    from cabinet_b200 import train_engine as te

    mob = backbone(mode).train()
    eng, rec = _record(monkeypatch, mob, te, te.TrainEngine, precision)
    x = torch.zeros(2, 3, 64, 64)
    y = eng.backbone_forward(x, input_grad)
    assert y.shape == (2, mob.out_channels, 2, 2)
    n_fwd = len(rec.calls)
    names = [c[0] for c in rec.calls]
    n_bn = sum(1 for m in mob.modules() if isinstance(m, torch.nn.BatchNorm2d))
    assert names.count("cabinet_bn_train_stats") == n_bn
    im2col = [a for n, a in rec.calls if n.startswith("cabinet_im2col_nchw")]
    if precision == "fp32":
        assert not im2col
    else:
        assert len(im2col) == 1
        a = im2col[0]
        assert a[5:8] == (3, 2, 1) and a[9] == 32   # k = 3, stride 2, pad 1; 27 columns padded to 32
    assert not [n for n in names if "attention" in n or "psp" in n or "stem_tc" in n or "cab_combine" in n]
    grads, dx = eng.backbone_backward(torch.zeros_like(y))
    bwd = [c for c in rec.calls[n_fwd:]]
    assert [n for n, _ in bwd].count("cabinet_bn_train_backward") == n_bn
    dgrad = [a for n, a in bwd if n == "cabinet_stem_dgrad"]
    if input_grad:
        assert len(dgrad) == 1 and dgrad[0][0] is None and dgrad[0][5] is None and dgrad[0][3] > 0   # dy7 = w7 = NULL
        assert dx is not None and dx.shape == x.shape
    else:
        assert not dgrad and dx is None
    trained = {id(p): n for n, p in mob.named_parameters() if not n.startswith("classifier")}
    assert set(grads) == set(trained), [trained[i] for i in set(trained) - set(grads)]


def test_cabinet_schedules_keep_the_7x7_footprint(monkeypatch):
    from cabinet_b200 import train_engine as te
    from cabinet_b200.synthetic import build_model

    net = build_model(5, "large").train()
    eng, rec = _record(monkeypatch, net, te, te.TrainEngine, "bf16")
    eng.forward(torch.zeros(1, 3, 64, 64))
    im2col = [a for n, a in rec.calls if n == "cabinet_im2col_nchw"]
    assert len(im2col) == 1 and im2col[0][5:8] == (7, 2, 3) and im2col[0][9] == 152
    assert "cabinet_stem3_tc" not in [n for n, _ in rec.calls]


# ---------------------------------------------------------------------------------------------------- the kernel
def test_stem3_compiles_without_spills_and_uses_tcgen05():
    log = _lib.CSRC / "build" / "stem_tc2.ptxas.log"
    if not log.is_file():
        pytest.skip("no ptxas log (the library was not built here)")
    bodies = {m.group(1): (m.group(2), m.group(3)) for m in re.finditer(
        r"Compiling entry function '(\w*stem\w*_kernel\w*)' for '(\w+)'(.*?)(?=Compiling entry function|\Z)",
        log.read_text(), flags=re.S)}
    names = [n for n in bodies if "stem3_tc_kernel" in n]
    assert len(names) == 1, list(bodies)
    arch, body = bodies[names[0]]
    assert arch == "sm_100a"
    assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in body, body
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not Path(cuobjdump).is_file():
        pytest.skip("cuobjdump is not installed")
    sass = subprocess.run([cuobjdump, "-sass", str(_lib.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    secs = [sec for sec in re.split(r"\n\s*Function : ", sass)[1:] if "stem3_tc_kernel" in sec.split("\n", 1)[0]]
    assert len(secs) == 1 and secs[0].count("UTCHMMA") == 3   # one M128 N16 K16 MMA per tap row

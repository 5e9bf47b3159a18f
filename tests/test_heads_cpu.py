"""No GPU: SpatialBranch / AttentionBranch / FeatureFusionModule / CABiNetOutput on their own -- validation, parameter
surface, engine housekeeping, their inference and training schedules against the recording double of the C-ABI, and the
compiled sb.conv1-only stem kernel (``stem_tc2_kernel`` at N = 64; the N = 80 instantiation CABiNet runs is unchanged)."""

import copy
import hashlib
import pickle
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from cabinet_b200 import (AttentionBranch, CABiNet, CABiNetOutput, ContextAggregationBlock, FeatureFusionModule,
                          MobileNetV3, SpatialBranch, _lib)
from cabinet_b200.constants import BACKBONE_CFGS
from cabinet_b200 import engine as engine_mod
from cabinet_b200.synthetic import build_model, state_dict_digest
from oracle.make_golden import MODEL_CASES
from tests.test_backbone_cpu import _record

GOLDEN = Path(__file__).resolve().parent / "golden"


def modules():
    torch.manual_seed(0)
    return {"sb": (SpatialBranch(), [(2, 3, 64, 64)]),
            "ab": (AttentionBranch(512, 128, 128, 19), [(2, 512, 8, 16)]),
            "ffm": (FeatureFusionModule(64 + 128, 128), [(2, 64, 16, 16), (2, 128, 16, 16)]),
            "head": (CABiNetOutput(128, 64, 19), [(2, 128, 16, 16)])}


# ---------------------------------------------------------------------------------------------------- validation
@pytest.mark.parametrize("kind", ["sb", "ab", "ffm", "head"])
def test_cpu_input_wrong_shape_and_dtype(kind):
    m, shapes = modules()[kind]
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(*[torch.zeros(s) for s in shapes])
    with pytest.raises(TypeError, match="float32, bfloat16 or float16"):
        m(*[torch.zeros(s, dtype=torch.float64) for s in shapes])
    bad = shapes[:-1] + [(shapes[-1][0], shapes[-1][1] + 8) + shapes[-1][2:]]   # channels off by 8
    with pytest.raises(ValueError):
        m(*[torch.zeros(s) for s in bad])
    with pytest.raises(ValueError):
        m(*[torch.zeros(s[1:]) for s in shapes])


@pytest.mark.parametrize("args,match", [((512, 128, 256, 19), "interplanes == outplanes"),
                                        ((512, 136, 136, 19), "interplanes % 16"),
                                        ((500, 128, 128, 19), "inplanes % 8")])
def test_attention_branch_widths(args, match):
    with pytest.raises(ValueError, match=match):
        AttentionBranch(*args)(torch.zeros(1, args[0], 4, 4))


def test_ffm_and_head_widths():
    with pytest.raises(ValueError, match="two multiples of 8"):
        FeatureFusionModule(64 + 128, 128)(torch.zeros(1, 60, 4, 4), torch.zeros(1, 132, 4, 4))
    with pytest.raises(ValueError, match="two multiples of 8"):
        FeatureFusionModule(64, 128)(torch.zeros(1, 64, 4, 4), torch.zeros(1, 0, 4, 4))
    with pytest.raises(ValueError, match="out_chan % 8"):
        FeatureFusionModule(64, 100)(torch.zeros(1, 32, 4, 4), torch.zeros(1, 32, 4, 4))
    with pytest.raises(ValueError, match="differ in N / h / w"):
        FeatureFusionModule(64, 64)(torch.zeros(1, 32, 4, 4), torch.zeros(1, 32, 4, 5))
    with pytest.raises(ValueError, match="differ in dtype"):
        FeatureFusionModule(64, 64)(torch.zeros(1, 32, 4, 4), torch.zeros(1, 32, 4, 4, dtype=torch.bfloat16))
    with pytest.raises(ValueError, match="in_chan % 8"):
        CABiNetOutput(100, 64, 19)(torch.zeros(1, 100, 4, 4))
    with pytest.raises(ValueError, match="mid_chan % 8"):
        CABiNetOutput(128, 60, 19)(torch.zeros(1, 128, 4, 4))


# ---------------------------------------------------------------------------------------------------- parameter surface
@pytest.mark.parametrize("name,mode,C,shape", MODEL_CASES)
def test_state_dict_unchanged(name, mode, C, shape):
    g = np.load(GOLDEN / f"model_{name}.npz")
    net = build_model(C, mode)
    assert state_dict_digest(net.state_dict()) == str(g["digest"])   # keys, order and values of the reference's
    for child, cls, args in (("sb", SpatialBranch, ()), ("ab", AttentionBranch, (net.attention_planes, 256, 256, C)),
                             ("ffm", FeatureFusionModule, (384, 256)), ("conv_out", CABiNetOutput, (256, 256, C))):
        keys = [k[len(child) + 1:] for k in net.state_dict() if k.startswith(child + ".")]
        assert list(cls(*args).state_dict()) == keys == list(getattr(net, child).state_dict()), child


def _with_engines(m):
    m.__dict__["_engine"], m.__dict__["_train_engine"] = object(), object()
    return m


@pytest.mark.parametrize("kind", ["sb", "ab", "ffm", "head"])
def test_deepcopy_pickle_and_to_drop_the_engines(kind):
    m = _with_engines(modules()[kind][0])
    for c in (copy.deepcopy(m), pickle.loads(pickle.dumps(m))):
        assert c.__dict__["_engine"] is None and c.__dict__["_train_engine"] is None
        assert c.precision == "bf16" and c.train_precision == "fp32"
    assert m.__dict__["_engine"] is not None
    m.float()
    assert m.__dict__["_engine"] is None and m.__dict__["_train_engine"] is None


def test_cabinet_drops_its_childrens_engines():
    net = CABiNet(5, mode="small")
    kids = (net.sb, net.ab, net.ffm, net.conv_out)
    for k in kids:
        _with_engines(k)
    c = copy.deepcopy(net)
    assert all(getattr(c, n).__dict__["_engine"] is None for n in ("sb", "ab", "ffm", "conv_out"))
    p = pickle.loads(pickle.dumps(net))
    assert all(getattr(p, n).__dict__["_engine"] is None for n in ("sb", "ab", "ffm", "conv_out"))
    net.float()
    assert all(k.__dict__["_engine"] is None and k.__dict__["_train_engine"] is None for k in kids)


# ---------------------------------------------------------------------------------------------------- dry runs
def _inference(monkeypatch, kind, precision, shapes):
    m = modules()[kind][0].eval()
    eng, rec = _record(monkeypatch, m, engine_mod, engine_mod.Engine, precision)
    layers = []
    run = eng._run
    monkeypatch.setattr(eng, "_run", lambda kernel, layer, *a: (layers.append(layer), run(kernel, layer, *a))[1])
    fwd = {"sb": eng.forward_sb, "ab": eng.forward_ab, "ffm": eng.forward_ffm, "head": eng.forward_head}[kind]
    ys = fwd(*[torch.zeros(s) for s in shapes])
    return m, eng, rec, layers, ys


@pytest.mark.parametrize("precision,W", [("bf16", 64), ("bf16", 70), ("fp32", 64)])
def test_inference_schedule_of_the_spatial_branch(monkeypatch, precision, W):
    m, eng, rec, layers, y = _inference(monkeypatch, "sb", precision, [(2, 3, 64, W)])
    assert set(engine_mod.Engine.SB_ATTRS) <= set(vars(eng)) and not hasattr(eng, "stem_tc2") and not hasattr(eng, "b1")
    assert y.shape == (2, 128, 8, -(-W // 8)) and y.dtype == torch.float32
    names = [c[0] for c in rec.calls]
    tc = precision == "bf16" and W % 4 == 0
    assert "cabinet_stem_tc2" not in names and "cabinet_stem_tc" not in names and "cabinet_stem3_tc" not in names
    assert layers.count("sb.conv1") == 1 and layers[0] == "sb.conv1"
    assert names[0] == ("cabinet_stem7_tc" if tc else "cabinet_conv2d_simt")
    assert layers == ["sb.conv1", "sb.conv2", "sb.conv3", "sb.conv_out", "sb.out"]
    assert eng.launches == len(names)
    if tc:
        a = dict(zip(("x", "N", "H", "W", "w", "y", "ld", "OH", "OW"), rec.calls[0][1]))
        assert (a["N"], a["H"], a["W"], a["ld"], a["OH"], a["OW"]) == (2, 64, W, 64, 32, W // 2)
        assert tuple(eng.stem_tc7.shape) == (7, 2, 2, 64, 8) and eng.stem_tc7.dtype == torch.bfloat16
    else:
        assert eng.stem_tc7 is None if precision == "fp32" else eng.stem_tc7 is not None


def test_stem7_weights_are_rows_0_to_63_of_the_fused_stem_pack(monkeypatch):
    net = build_model(5, "small").eval()
    eng7, _ = _record(monkeypatch, net.sb, engine_mod, engine_mod.Engine, "bf16")
    eng, _ = _record(monkeypatch, net, engine_mod, engine_mod.Engine, "bf16")
    assert torch.equal(eng7.stem_tc7, eng.stem_tc2[:, :, :, :64].contiguous())


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_inference_schedules_of_the_attention_branch_ffm_and_head(monkeypatch, precision):
    m, eng, rec, layers, (low, high) = _inference(monkeypatch, "ab", precision, [(2, 512, 8, 16)])
    assert low.shape == (2, 128, 8, 16) and high.shape == (2, 19, 8, 16)
    assert not hasattr(eng, "sb1") and not hasattr(eng, "ffm_blk") and not hasattr(eng, "blocks")
    assert layers[0] == "ab.in" and layers[1] == "ab.conva" and layers[-2:] == ["ab.low", "ab.high"]
    for n in ("ab.convb", "ab.b1", "ab.b4"):
        assert layers.count(n) == 1, n
    assert "low_up" not in layers and "high_up" not in layers and not [n for n in layers if n.startswith(("sb.", "ffm"))]
    names = [c[0] for c in rec.calls]
    b1 = [a for (n, a), l in zip(rec.calls, layers) if l == "ab.b1"][0]
    resample = [a for n, a in rec.calls if n == "cabinet_resample_sep"]
    assert len(resample) == 3
    # x lands in channels [0:512] of the 640-channel b1 input, which b1 reads whole
    assert resample[0][8:11] == (8 * 16 * 640, 16 * 640, 640) and resample[0][6] == b1[0]

    m, eng, rec, layers, y = _inference(monkeypatch, "ffm", precision, [(2, 64, 16, 16), (2, 128, 16, 16)])
    assert y.shape == (2, 128, 16, 16)
    names = [c[0] for c in rec.calls]
    assert layers == ["ffm.in_sp", "ffm.in_cp", "ffm.convblk", "ffm.gap", "ffm.gate", "ffm.gate", "ffm.gate", "ffm.out"]
    assert names[3:7] == ["cabinet_channel_sum", "cabinet_gate_fc", "cabinet_gate_fc", "cabinet_scale_act"]
    assert rec.calls[6][1][-2] == 1   # plus_one: feat * atten + feat
    sp, cp = [a for n, a in rec.calls[:2]]
    assert cp[6] - sp[6] == 64 * (2 if precision == "bf16" else 4)   # fcp starts at channel 64 of the same pixel
    assert eng.launches == len(names) + 1   # + the memset of the pooling sums / scratch

    m, eng, rec, layers, y = _inference(monkeypatch, "head", precision, [(2, 128, 16, 16)])
    assert y.shape == (2, 19, 16, 16)
    assert layers == ["conv_out.in", "conv_out.conv", "conv_out.conv_out", "conv_out.out"]
    assert "cabinet_gate_scale_weights" not in [c[0] for c in rec.calls]


@pytest.mark.parametrize("precision", ["bf16", "fp32", "fp16"])
@pytest.mark.parametrize("input_grad", [False, True])
def test_training_schedule_of_the_spatial_branch(monkeypatch, precision, input_grad):
    from cabinet_b200 import train_engine as te

    m = SpatialBranch().train()
    eng, rec = _record(monkeypatch, m, te, te.TrainEngine, precision)
    x = torch.zeros(2, 3, 64, 64)
    (y,), record = eng.module_forward([x], [input_grad])
    assert y.shape == (2, 128, 8, 8)
    n_fwd = len(rec.calls)
    names = [c[0] for c in rec.calls]
    assert names.count("cabinet_bn_train_stats") == 4
    im2col = [a for n, a in rec.calls if n.startswith("cabinet_im2col_nchw")]
    if precision == "fp32":
        assert not im2col
    else:
        assert len(im2col) == 1 and im2col[0][5:8] == (7, 2, 3) and im2col[0][9] == 152
    assert not [n for n in names if "stem_tc" in n or "stem3" in n or "stem7" in n]
    grads, dxs = eng.module_backward(record, [torch.zeros_like(y)], [x.dtype])
    bwd = rec.calls[n_fwd:]
    assert [n for n, _ in bwd].count("cabinet_bn_train_backward") == 4
    dgrad = [a for n, a in bwd if n == "cabinet_stem_dgrad"]
    if input_grad:
        assert len(dgrad) == 1 and dgrad[0][2] is None and dgrad[0][6] is None and dgrad[0][1] > 0   # dy3 = w3 = NULL
        assert dxs[0] is not None and dxs[0].shape == x.shape
    else:
        assert not dgrad and dxs == [None]
    assert set(grads) == {id(p) for p in m.parameters()}


@pytest.mark.parametrize("used", ["both", "low", "high"])
def test_training_schedule_of_the_attention_branch(monkeypatch, used):
    from cabinet_b200 import train_engine as te

    m = AttentionBranch(512, 128, 128, 19).train()
    eng, rec = _record(monkeypatch, m, te, te.TrainEngine, "bf16")
    x = torch.zeros(2, 512, 8, 16)
    (low, high), record = eng.module_forward([x], [True])
    n_fwd = len(rec.calls)
    dys = [torch.zeros_like(low) if used != "high" else None, torch.zeros_like(high) if used != "low" else None]
    grads, (dx,) = eng.module_backward(record, dys, [x.dtype])
    bwd = [n for n, _ in rec.calls[n_fwd:]]
    n_bn = sum(1 for mm in m.modules() if isinstance(mm, torch.nn.BatchNorm2d))
    assert bwd.count("cabinet_bn_train_backward") == n_bn - (1 if used == "low" else 0)   # b2: only on the high path
    unused = {"low": ("b1.", "b2.", "b4."), "high": ("convb.",), "both": ()}[used]
    assert set(grads) == {id(p) for n, p in m.named_parameters() if not n.startswith(unused)}
    assert dx is not None and dx.shape == x.shape


def test_training_schedules_of_the_ffm_and_head(monkeypatch):
    from cabinet_b200 import train_engine as te

    m = FeatureFusionModule(64 + 128, 128).train()
    eng, rec = _record(monkeypatch, m, te, te.TrainEngine, "bf16")
    fsp, fcp = torch.zeros(2, 64, 16, 16), torch.zeros(2, 128, 16, 16)
    (y,), record = eng.module_forward([fsp, fcp], [False, True])
    assert y.shape == (2, 128, 16, 16)
    grads, (dsp, dcp) = eng.module_backward(record, [torch.zeros_like(y)], [fsp.dtype, fcp.dtype])
    assert dsp is None and dcp is not None and dcp.shape == fcp.shape
    assert set(grads) == {id(p) for p in m.parameters()}
    assert [n for n, _ in rec.calls].count("cabinet_gate_mlp_backward") == 1

    m = CABiNetOutput(128, 64, 19).train()
    eng, rec = _record(monkeypatch, m, te, te.TrainEngine, "fp32")
    (y,), record = eng.module_forward([torch.zeros(2, 128, 16, 16)], [False])
    assert y.shape == (2, 19, 16, 16)
    grads, dxs = eng.module_backward(record, [torch.zeros_like(y)], [torch.float32])
    assert dxs == [None] and set(grads) == {id(p) for p in m.parameters()}


def test_two_calls_before_one_backward_keep_their_own_tapes(monkeypatch):
    from cabinet_b200 import train_engine as te

    m = SpatialBranch().train()
    eng, rec = _record(monkeypatch, m, te, te.TrainEngine, "bf16")
    x1, x2 = torch.zeros(2, 3, 64, 64), torch.zeros(1, 3, 32, 48)
    (y1,), r1 = eng.module_forward([x1], [True])
    n1 = len(rec.calls)
    (y2,), r2 = eng.module_forward([x2], [True])
    assert r1[0] is not r2[0] and r1[0] and r2[0] and eng.tape == []
    n_fwd = len(rec.calls)
    _, (dx2,) = eng.module_backward(r2, [torch.zeros_like(y2)], [x2.dtype])
    _, (dx1,) = eng.module_backward(r1, [torch.zeros_like(y1)], [x1.dtype])
    assert dx1.shape == x1.shape and dx2.shape == x2.shape   # each backward ran its own call's tape
    dgrad = [a for n, a in rec.calls[n_fwd:] if n == "cabinet_stem_dgrad"]
    assert [a[8:11] for a in dgrad] == [(1, 32, 48), (2, 64, 64)] and n_fwd > n1


class _MyMob(MobileNetV3):
    pass


class _MyBlock(ContextAggregationBlock):
    pass


class _MySB(SpatialBranch):
    pass


class _MyAB(AttentionBranch):
    pass


class _MyFFM(FeatureFusionModule):
    pass


class _MyHead(CABiNetOutput):
    pass


@pytest.mark.parametrize("cls,args,fwd,shapes", [
    (_MyMob, (BACKBONE_CFGS["small"], "small"), "forward_backbone", [(1, 3, 64, 64)]),
    (_MyBlock, (256, 128), "forward_block", [(1, 256, 8, 16)]),
    (_MySB, (), "forward_sb", [(1, 3, 64, 64)]),
    (_MyAB, (512, 128, 128, 19), "forward_ab", [(1, 512, 8, 16)]),
    (_MyFFM, (64 + 128, 128), "forward_ffm", [(1, 64, 16, 16), (1, 128, 16, 16)]),
    (_MyHead, (128, 64, 19), "forward_head", [(1, 128, 16, 16)]),
])
def test_engines_over_subclasses_run_the_standalone_schedule(monkeypatch, cls, args, fwd, shapes):
    from cabinet_b200 import train_engine as te

    m = cls(*args).eval()
    eng, rec = _record(monkeypatch, m, engine_mod, engine_mod.Engine, "bf16")
    assert not hasattr(eng, "stem_tc2") and eng.n_classes == 0
    getattr(eng, fwd)(*[torch.zeros(s) for s in shapes])
    assert rec.calls and not [n for n, _ in rec.calls if n in ("cabinet_stem_tc2", "cabinet_upsample_logits_nchw")]
    if fwd not in ("forward_backbone", "forward_block"):
        teng, trec = _record(monkeypatch, m.train(), te, te.TrainEngine, "bf16")
        ys, record = teng.module_forward([torch.zeros(s) for s in shapes], [True] * len(shapes))
        grads, dxs = teng.module_backward(record, [torch.zeros_like(y) for y in ys], [torch.float32] * len(shapes))
        assert set(grads) == {id(p) for p in m.parameters()}


# ---------------------------------------------------------------------------------------------------- the kernel
def _sass_functions():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not _lib.LIB_PATH.is_file() or not Path(cuobjdump).is_file():
        pytest.skip("no library or no cuobjdump here")
    sass = subprocess.run([cuobjdump, "-sass", str(_lib.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    return {sec.split("\n", 1)[0].strip(): sec for sec in re.split(r"\n\s*Function : ", sass)[1:]}


def test_stem7_compiles_without_spills_and_uses_tcgen05():
    log = _lib.CSRC / "build" / "stem_tc2.ptxas.log"
    if not log.is_file():
        pytest.skip("no ptxas log (the library was not built here)")
    bodies = {m.group(1): (m.group(2), m.group(3)) for m in re.finditer(
        r"Compiling entry function '(\w*stem\w*_kernel\w*)' for '(\w+)'(.*?)(?=Compiling entry function|\Z)",
        log.read_text(), flags=re.S)}
    names = [n for n in bodies if "stem_tc2_kernelILi64E" in n]
    assert len(names) == 1, list(bodies)
    arch, body = bodies[names[0]]
    assert arch == "sm_100a"
    assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in body, body
    secs = [s for n, s in _sass_functions().items() if "stem_tc2_kernelILi64E" in n]
    assert len(secs) == 1 and secs[0].count("UTCHMMA") == 14   # 7 tap rows x 2 K halves of M128 N64 K16


# the instruction stream of stem_tc2_kernel (CABiNet's fused stems) as CUDA 12.9's nvcc compiled it before the kernel
# was templated on its output width: sha256 over the instructions (addresses and encodings stripped), and their count
STEM_TC2_SASS = ("876dcf50079d0cd523d9718d33ef7caf6e7377f1fca2f6f17900e5ea4151d137", 992)


def test_stem_tc2_kernel_sass_is_unchanged():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).is_file() or "release 12.9" not in subprocess.run([nvcc, "--version"], capture_output=True,
                                                                          text=True).stdout:
        pytest.skip("the recorded instruction stream is CUDA 12.9's")
    secs = [s for n, s in _sass_functions().items() if "stem_tc2_kernelILi80E" in n]
    assert len(secs) == 1
    ins = [m.group(1).strip() for m in re.finditer(r"/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;", secs[0])]
    assert (hashlib.sha256("\n".join(ins).encode()).hexdigest(), len(ins)) == STEM_TC2_SASS

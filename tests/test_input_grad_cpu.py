"""CPU: gradients with respect to the input image, without a GPU.

The training schedule runs against the recording double of the C-ABI (tests/test_train_fp16_cpu.py), with every tape
entry wrapped to record the calls its backward issues (tests/test_train_freeze_cpu.py).

* ``x`` without grad: no ``cabinet_stem_dgrad`` call;
* train mode, ``x`` requires grad: the default schedule plus exactly one ``cabinet_stem_dgrad``, after both stems' BN
  backward calls (Large and Small, fp32 / bf16 / fp16);
* eval mode, every parameter frozen: no weight gradient, ``col_sum`` or ``bn_train_*``, one ``bn_frozen_backward`` per
  BN (dz only), one ``cabinet_stem_dgrad``, running statistics untouched;
* routing of ``CABiNet.forward``: eval mode reaches ``TrainStep`` only with grad mode on and ``x.requires_grad``;
* ``cabinet_stem_dgrad`` rejects bad arguments before any CUDA call; its kernels compile for sm_100a without spills and
  the 2-byte instantiations issue tcgen05.mma (UTCHMMA).
"""

import ctypes
import re
import shutil
import subprocess
from collections import Counter
from pathlib import Path

import pytest
import torch
from torch import nn

from cabinet_b200 import _lib
from cabinet_b200.synthetic import build_model
from tests.test_train_fp16_cpu import RecordingLib
from tests.test_train_freeze_cpu import SCHEDULE, SHAPE, WGRAD, _owned, bns, names

STEM = "cabinet_stem_dgrad"


def record(monkeypatch, input_grad, prepare=None, precision="bf16", mode="large", classes=5, shape=SHAPE):
    """-> (model, forward calls, backward calls, [(parameter ids of a tape entry, indices of its backward calls)], grads,
    engine)."""
    from cabinet_b200 import train_engine as te

    rec = RecordingLib()
    monkeypatch.setattr(_lib, "load", lambda: rec)
    monkeypatch.setattr(te.TrainEngine, "stream", property(lambda self: None))
    model = build_model(classes, mode).train()
    if prepare is not None:
        prepare(model)

    class P:
        is_cuda = True
        device = torch.device("cpu")

    real_next = next
    monkeypatch.setattr(te, "next", lambda it: P, raising=False)
    eng = te.TrainEngine(model, precision)
    monkeypatch.setattr(te, "next", real_next, raising=False)
    final, aux = eng.forward(torch.zeros(shape), input_grad=input_grad)
    fwd = list(rec.calls)
    n0 = len(rec.calls)
    entries = []

    def wrap(fn):
        entry = [_owned(fn), []]
        entries.append(entry)

        def run(g):
            n = len(rec.calls)
            fn(g)
            entry[1].extend(range(n - n0, len(rec.calls) - n0))

        return run

    eng.tape = [wrap(fn) for fn in eng.tape]
    grads = eng.backward(torch.zeros_like(final), torch.zeros_like(aux))
    return model, fwd, rec.calls[n0:], entries, grads, eng


def stem_bns(model):
    return [model.sb.conv1.bn, model.mobile.features[0][1]]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_no_input_grad_no_stem_dgrad(monkeypatch, precision):
    _, fwd, bwd, _, _, eng = record(monkeypatch, False, precision=precision)
    assert STEM not in names(fwd) + names(bwd)
    assert eng.dx is None


@pytest.mark.parametrize("mode,classes,shape", [("large", 5, SHAPE), ("small", 8, (2, 3, 64, 96))])
@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp16"])
def test_train_mode_adds_one_stem_dgrad(monkeypatch, mode, classes, shape, precision):
    model, fwd, bwd, entries, _, eng = record(monkeypatch, True, precision=precision, mode=mode, classes=classes, shape=shape)
    counts = names(fwd) + names(bwd)
    assert counts[STEM] == 1
    del counts[STEM]
    assert dict(counts) == SCHEDULE[f"{mode}-{precision}"]
    (i_stem,) = [i for i, (n, _) in enumerate(bwd) if n == STEM]
    for bn in stem_bns(model):
        owned = [idx for ids, idx in entries if id(bn.weight) in ids]
        assert owned and owned[0], bn
        assert max(owned[0]) < i_stem
        assert all(bwd[i][0] in ("cabinet_bn_train_backward", "cabinet_add") for i in owned[0])
    args = bwd[i_stem][1]
    N, _, H, W = shape
    # (dy7, ld7, dy3, ld3, dtype, w7, w3, dx, N, H, W, OH, OW, stream)
    assert args[0] is not None and args[2] is not None
    assert (args[1], args[3]) == (64, 16)
    assert args[4] == {"fp32": _lib.F32, "bf16": _lib.BF16, "fp16": _lib.F16}[precision]
    assert args[5] == model.sb.conv1.conv.weight.data_ptr() and args[6] == model.mobile.features[0][0].weight.data_ptr()
    assert args[7] == eng.dx.data_ptr() and eng.dx.shape == (N, 3, H, W) and eng.dx.dtype == torch.float32
    assert args[8:13] == (N, H, W, (H - 1) // 2 + 1, (W - 1) // 2 + 1)


def _eval_frozen(model):
    model.eval()
    for p in model.parameters():
        p.requires_grad_(False)


@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp16"])
def test_eval_frozen_attack_step(monkeypatch, precision):
    before = {}

    def prepare(model):
        _eval_frozen(model)
        before.update({k: v.clone() for k, v in model.state_dict().items()})

    model, fwd, bwd, _, grads, _ = record(monkeypatch, True, prepare, precision)
    nf, nb = names(fwd), names(bwd)
    assert not any(nb[k] for k in WGRAD) and nb["cabinet_col_sum"] == 0
    assert not any(n.startswith("cabinet_bn_train") for n in nf + nb)
    assert nf["cabinet_bn_frozen_stats"] == nb["cabinet_bn_frozen_backward"] == len(bns(model))
    for name, args in bwd:
        if name == "cabinet_bn_frozen_backward":   # dz only: no parameter reduction
            assert args[7] is None and args[8] is None and args[9] is not None and args[14] is None
    assert nb[STEM] == 1
    assert grads == {}
    for k, v in model.state_dict().items():
        assert torch.equal(v, before[k]), k


def test_eval_frozen_aux_only_skips_the_spatial_stem(monkeypatch):
    """Only the auxiliary output in the loss: sb.conv1 gets no gradient, cabinet_stem_dgrad gets a NULL dy7."""
    from cabinet_b200 import train_engine as te

    rec = RecordingLib()
    monkeypatch.setattr(_lib, "load", lambda: rec)
    monkeypatch.setattr(te.TrainEngine, "stream", property(lambda self: None))
    model = build_model(5, "large")
    _eval_frozen(model)

    class P:
        is_cuda = True
        device = torch.device("cpu")

    real_next = next
    monkeypatch.setattr(te, "next", lambda it: P, raising=False)
    eng = te.TrainEngine(model, "bf16")
    monkeypatch.setattr(te, "next", real_next, raising=False)
    _, aux = eng.forward(torch.zeros(SHAPE), input_grad=True)
    n0 = len(rec.calls)
    eng.backward(None, torch.zeros_like(aux))
    (args,) = [a for n, a in rec.calls[n0:] if n == STEM]
    assert args[0] is None and args[2] is not None


# ----------------------------------------------------------------------------- routing of CABiNet.forward
@pytest.fixture
def routed(monkeypatch):
    """A model whose engines are stand-ins: -> (model, list of 'train' / 'infer' per forward call)."""
    from cabinet_b200 import train_engine as te

    model = build_model(5, "large")
    seen = []

    class Infer:
        def forward(self, x, out_dtype):
            seen.append("infer")
            return x, x

    monkeypatch.setattr(type(model), "_check_input", lambda self, x, inference_only=True: None)
    monkeypatch.setattr(type(model), "engine", lambda self: Infer())
    monkeypatch.setattr(type(model), "train_engine", lambda self: None)
    monkeypatch.setattr(te.TrainStep, "apply", lambda *a: seen.append("train") or (a[3], a[3]))
    return model, seen


def test_routing_eval(routed):
    model, seen = routed
    model.eval()
    x = torch.zeros(1, 3, 8, 8, requires_grad=True)
    model(x)
    assert seen == ["train"]
    with torch.no_grad():
        model(x)
    with torch.inference_mode():
        model(torch.zeros(1, 3, 8, 8))
    model(torch.zeros(1, 3, 8, 8))
    model(x.detach())
    assert seen == ["train"] + ["infer"] * 4


def test_routing_train(routed):
    model, seen = routed
    model.train()
    model(torch.zeros(1, 3, 8, 8))
    model(torch.zeros(1, 3, 8, 8, requires_grad=True))
    assert seen == ["train", "train"]


# ----------------------------------------------------------------------------- the entry point
def _lib_or_skip():
    if not _lib.LIB_PATH.is_file():
        pytest.skip("libcabinet_b200.so is not built")
    return _lib.load()


def test_stem_dgrad_rejects_bad_arguments():
    lib = _lib_or_skip()
    p = ctypes.c_void_p(256)   # never dereferenced: every case fails its argument check first
    good = [p, 64, p, 16, _lib.BF16, p, p, p, 2, 70, 100, 35, 50, None]

    def call(**kw):
        a = list(good)
        for k, v in kw.items():
            a[int(k[1:])] = v
        return lib.cabinet_stem_dgrad(*a)

    for dt in (3, 7, -1):
        assert call(a4=dt) == 1 and "element type" in lib.cabinet_last_error().decode()
    assert call(a0=None, a2=None) == 1 and "both output gradients are NULL" in lib.cabinet_last_error().decode()
    assert call(a7=None) == 1 and "NULL dx" in lib.cabinet_last_error().decode()
    for kw in (dict(a11=36), dict(a12=49), dict(a11=34), dict(a9=0), dict(a10=0), dict(a8=-1)):
        assert call(**kw) == 1, kw
        assert "bad sizes" in lib.cabinet_last_error().decode(), kw
    for kw in (dict(a1=32), dict(a1=68), dict(a3=8), dict(a5=None), dict(a6=None), dict(a0=ctypes.c_void_p(258))):
        assert call(**kw) == 1, kw
        assert "stem_dgrad" in lib.cabinet_last_error().decode(), kw
    assert call(a4=_lib.F32, a1=66) == 1   # fp32: 16-byte pixels need ld % 4 == 0
    assert call(a8=0) == 0                  # an empty batch is a no-op


def test_stem_dgrad_compiles_without_spills_and_uses_tcgen05():
    log = _lib.CSRC / "build" / "stem_dgrad.ptxas.log"
    if not log.is_file():
        pytest.skip("no ptxas log (the library was not built here)")
    found = Counter()
    for m in re.finditer(r"Compiling entry function '(\w*stem_dgrad\w+)' for '(\w+)'(.*?)(?=Compiling entry function|\Z)",
                         log.read_text(), flags=re.S):
        name, arch, body = m.groups()
        assert arch == "sm_100a", name
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in body, (name, body)
        found["tc" if "tc_kernel" in name else "f32"] += 1
    assert found == Counter({"tc": 2, "f32": 1}), found
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not Path(cuobjdump).is_file():
        pytest.skip("cuobjdump is not installed")
    sass = subprocess.run([cuobjdump, "-sass", str(_lib.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    types = []
    for sec in re.split(r"\n\s*Function : ", sass)[1:]:
        name = sec.split("\n", 1)[0]
        if "stem_dgrad_tc_kernel" in name:
            assert "UTCHMMA" in sec, name
            types.append("bf16" if "bfloat16" in name else "fp16" if "6__half" in name else name)
    assert sorted(types) == ["bf16", "fp16"], types

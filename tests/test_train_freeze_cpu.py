"""CPU: frozen parameters and eval-mode BatchNorm in the training step, without a GPU.

The schedule runs against the recording double of the C-ABI (tests/test_train_fp16_cpu.py).  Every tape entry is
wrapped to record the calls its backward issues; the layer an entry belongs to is read from its closure (the module or
parameters it captured).

* nothing frozen: the calls per entry point of the step before frozen modules were supported
  (``tests/golden/train_schedule_calls.json``), no new entry point, one train-BN stats / backward per BN, one weight
  gradient per convolution;
* all BN eval: ``bn_frozen_stats`` / ``bn_frozen_backward`` once per BN, ``bn_train_*`` never, no
  ``num_batches_tracked`` increment, the running statistics untouched;
* backbone frozen: one weight gradient per trainable convolution, no backward call for any backbone layer, gradients
  for exactly the trainable parameters;
* only ``conv_out.conv_out`` trainable: the final-logit adjoint and that layer's weight gradient, nothing else;
* both new entry points reject an unknown element type and bad sizes; their kernels compile for sm_100a without spills.
"""

import ctypes
import json
import re
from collections import Counter
from pathlib import Path

import pytest
import torch
from torch import nn

from cabinet_b200 import _lib
from cabinet_b200.synthetic import build_model
from tests.test_train_fp16_cpu import RecordingLib

SHAPE = (2, 3, 256, 512)   # Large: 128-token attention at 1/32, so the tensor-core attention runs too
WGRAD = {"cabinet_conv_wgrad", "cabinet_conv_wgrad_tc", "cabinet_conv_wgrad_tc_dt", "cabinet_dwconv_wgrad"}
NEW = {"cabinet_bn_frozen_stats", "cabinet_bn_frozen_backward"}


def _owned(fn):
    """ids of the parameters a tape entry's closure captured (a layer's module or its parameters)."""
    ids = set()
    for cell in fn.__closure__ or ():
        try:
            v = cell.cell_contents
        except ValueError:
            continue
        if isinstance(v, nn.Parameter):
            ids.add(id(v))
        elif isinstance(v, nn.Module):
            ids.update(id(p) for p in v.parameters())
    return ids


def record(monkeypatch, freeze=None, precision="bf16", mode="large", classes=5, shape=SHAPE):
    """-> (model, forward calls, backward calls, [(parameter ids of a tape entry, its backward calls)], gradients)."""
    from cabinet_b200 import train_engine as te

    rec = RecordingLib()
    monkeypatch.setattr(_lib, "load", lambda: rec)
    monkeypatch.setattr(te.TrainEngine, "stream", property(lambda self: None))
    model = build_model(classes, mode).train()
    if freeze is not None:
        freeze(model)

    class P:
        is_cuda = True
        device = torch.device("cpu")

    real_next = next
    monkeypatch.setattr(te, "next", lambda it: P, raising=False)
    eng = te.TrainEngine(model, precision)
    monkeypatch.setattr(te, "next", real_next, raising=False)
    final, aux = eng.forward(torch.zeros(shape))
    fwd = list(rec.calls)
    entries = []

    def wrap(fn):
        entry = [_owned(fn), []]
        entries.append(entry)

        def run(g):
            n = len(rec.calls)
            fn(g)
            entry[1].extend(name for name, _ in rec.calls[n:])

        return run

    eng.tape = [wrap(fn) for fn in eng.tape]
    n0 = len(rec.calls)
    grads = eng.backward(torch.zeros_like(final), torch.zeros_like(aux))
    return model, fwd, rec.calls[n0:], entries, grads


def bns(model, under=""):
    return [m for n, m in model.named_modules() if isinstance(m, nn.BatchNorm2d) and n.startswith(under)]


def names(calls):
    return Counter(n for n, _ in calls)


def gate_convs(model):
    return {id(model.ffm.conv1.weight), id(model.ffm.conv2.weight)}  # FFM attention: gate_mlp_backward, not a conv


def conv_weights(model, trainable_only=True):
    skip = gate_convs(model)
    return [m.weight for n, m in model.named_modules() if isinstance(m, nn.Conv2d) and not n.startswith("mobile.classifier")
            and id(m.weight) not in skip and (m.weight.requires_grad or not trainable_only)]


# Calls per entry point of one default step (forward + backward), recorded before eval-mode BN and frozen parameters
# were supported: with nothing frozen the schedule must stay exactly this.
SCHEDULE = json.loads((Path(__file__).resolve().parent / "golden" / "train_schedule_calls.json").read_text())


@pytest.mark.parametrize("mode,classes,shape", [("large", 5, SHAPE), ("small", 8, (2, 3, 64, 96))])
@pytest.mark.parametrize("precision", ["fp32", "bf16", "fp16"])
def test_nothing_frozen_calls_per_entry_point(monkeypatch, mode, classes, shape, precision):
    _, fwd, bwd, _, _ = record(monkeypatch, precision=precision, mode=mode, classes=classes, shape=shape)
    assert dict(names(fwd) + names(bwd)) == SCHEDULE[f"{mode}-{precision}"]


def test_nothing_frozen_keeps_the_schedule(monkeypatch):
    model, fwd, bwd, _, grads = record(monkeypatch)
    nf, nb = names(fwd), names(bwd)
    assert not (set(nf) | set(nb)) & NEW
    n_bn = len(bns(model))
    assert nf["cabinet_bn_train_stats"] == nb["cabinet_bn_train_backward"] == n_bn
    assert sum(nb[k] for k in WGRAD) == len(conv_weights(model))
    assert set(grads) == {id(p) for n, p in model.named_parameters() if not n.startswith("mobile.classifier")}


def _all_bn_eval(model):
    for m in bns(model):
        m.eval()


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_all_bn_eval(monkeypatch, precision):
    before = {}

    def freeze(model):
        _all_bn_eval(model)
        before.update({k: v.clone() for k, v in model.state_dict().items()})

    model, fwd, bwd, _, grads = record(monkeypatch, freeze, precision)
    nf, nb = names(fwd), names(bwd)
    n_bn = len(bns(model))
    assert nf["cabinet_bn_frozen_stats"] == nb["cabinet_bn_frozen_backward"] == n_bn
    assert nf["cabinet_bn_train_stats"] == nb["cabinet_bn_train_backward"] == 0
    for k, v in model.state_dict().items():   # num_batches_tracked and the running statistics: not touched
        assert torch.equal(v, before[k]), k
    # every BN's parameters and input need a gradient: both reductions and dz in the one call
    for name, args in bwd:
        if name == "cabinet_bn_frozen_backward":
            assert args[7] is not None and args[8] is not None and args[9] is not None
    assert sum(nb[k] for k in WGRAD) == len(conv_weights(model))
    assert set(grads) == {id(p) for n, p in model.named_parameters() if not n.startswith("mobile.classifier")}


def _freeze_backbone(model):
    for p in model.mobile.parameters():
        p.requires_grad_(False)
    for m in bns(model, "mobile"):
        m.eval()


def test_backbone_frozen(monkeypatch):
    model, fwd, bwd, entries, grads = record(monkeypatch, _freeze_backbone)
    backbone = {id(p) for p in model.mobile.parameters()}
    nb = names(bwd)
    assert sum(nb[k] for k in WGRAD) == len(conv_weights(model)) == len(
        [w for w in conv_weights(model, False) if id(w) not in backbone])
    assert nb["cabinet_bn_frozen_backward"] == 0   # the backbone's eval BNs lead to no trainable parameter
    assert nb["cabinet_bn_train_backward"] == len(bns(model)) - len(bns(model, "mobile"))
    n_backbone_entries = 0
    for owned, calls in entries:
        if owned & backbone:
            n_backbone_entries += 1
            assert calls == [], calls
    assert n_backbone_entries > 40
    assert set(grads) == {id(p) for p in model.parameters() if p.requires_grad}
    assert not set(grads) & backbone
    nf = names(fwd)
    assert nf["cabinet_bn_frozen_stats"] == len(bns(model, "mobile"))


def test_only_the_last_conv_trainable(monkeypatch):
    def freeze(model):
        for n, p in model.named_parameters():
            p.requires_grad_(n == "conv_out.conv_out.weight")

    model, _, bwd, entries, grads = record(monkeypatch, freeze)
    assert set(grads) == {id(model.conv_out.conv_out.weight)}
    # the final logits' adjoint (one resampling call) and the weight gradient of the fp32 class map's convolution
    assert names(bwd) == Counter({"cabinet_resample_sep": 1, "cabinet_conv_wgrad": 1}), names(bwd)
    owner = [calls for owned, calls in entries if id(model.conv_out.conv_out.weight) in owned]
    assert owner == [["cabinet_conv_wgrad"]]


def test_nothing_trainable_issues_no_backward(monkeypatch):
    def freeze(model):
        for p in model.parameters():
            p.requires_grad_(False)

    _, _, bwd, _, grads = record(monkeypatch, freeze)
    assert bwd == [] and grads == {}


def _lib_or_skip():
    if not _lib.LIB_PATH.is_file():
        pytest.skip("libcabinet_b200.so is not built")
    return _lib.load()


def test_new_entry_points_reject_bad_arguments():
    lib = _lib_or_skip()
    p = ctypes.c_void_p(256)   # never dereferenced: every case fails its argument check first
    # (dy, lddy, z, ldz, dtype, stats, act, dgamma, dbeta, dz, lddz, M, C, accumulate, scratch, stream)
    good = [p, 64, p, 64, _lib.BF16, p, 0, p, p, p, 64, 128, 64, 0, p, None]

    def bwd(**kw):
        a = list(good)
        for k, v in kw.items():
            a[int(k[1:])] = v
        return lib.cabinet_bn_frozen_backward(*a)

    for dt in (3, 7, -1):
        assert bwd(a4=dt) == 1 and "element type" in lib.cabinet_last_error().decode()
    bad = [dict(a11=0), dict(a12=0), dict(a12=-8), dict(a1=32), dict(a3=32), dict(a10=32), dict(a0=None),
           dict(a2=None), dict(a5=None), dict(a7=None, a8=None, a9=None), dict(a14=None)]
    for kw in bad:
        assert bwd(**kw) == 1, kw
        assert "bn_frozen_backward: bad arguments" in lib.cabinet_last_error().decode(), kw
    for a in ([p, p, p, p, 1e-5, 0, p, None], [p, p, None, p, 1e-5, 8, p, None], [p, p, p, p, 1e-5, 8, None, None],
              [p, p, p, p, -1.0, 8, p, None]):
        assert lib.cabinet_bn_frozen_stats(*a) == 1
        assert "bn_frozen_stats: bad arguments" in lib.cabinet_last_error().decode()


def test_frozen_bn_kernels_compile_without_spills():
    log = _lib.CSRC / "build" / "train.ptxas.log"
    if not log.is_file():
        pytest.skip("no ptxas log (the library was not built here)")
    text = log.read_text()
    found = Counter()
    for m in re.finditer(r"Compiling entry function '(\w*bn_frozen_\w+)' for '(\w+)'(.*?)(?=Compiling entry function|\Z)",
                         text, flags=re.S):
        name, arch, body = m.groups()
        assert arch == "sm_100a", name
        assert "0 bytes spill stores, 0 bytes spill loads" in body, (name, body)
        for tag, t in (("If", "fp32"), ("I13__nv_bfloat16", "bf16"), ("I6__half", "fp16")):
            if "bwd" in name and tag in name:
                found[t] += 1
        if "stats" in name:
            found["stats"] += 1
    # scalar and vector kernels, with and without the reduction, in each of the three types
    assert found == Counter({"fp32": 4, "bf16": 4, "fp16": 4, "stats": 1}), found

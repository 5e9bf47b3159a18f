"""CPU: the variant census of the training step's elementwise and reduction kernels.

The step runs against the recording double of the C-ABI (``tests/test_train_fp16_cpu.py``) for Large and Small in
fp32, bf16 and fp16, and for the freeze settings of ``tests/test_train_freeze_cpu.py``.  Every call to an entry point
of ``tests/train_variants.py`` gets its variant key (the inputs of its host dispatch).

* every recorded key has a case in the GPU replay matrix of ``tests/test_gpu_train_variants.py``, so a schedule change
  that reaches a new kernel path fails here until that path is tested on the GPU;
* the documented preconditions hold: ``ld >= C`` for every strided operand, dense ``g``, ``x``, ``r``, ``dg``, ``dx``,
  ``dr`` for ``cab_combine_backward`` and dense rows for ``softmax_backward`` (their ABI has no stride);
* ``cab_combine_backward`` overwrites ``dg`` and ``dr``: the gradient regions it is given are first writes.
"""

from collections import defaultdict

import pytest
import torch

from cabinet_b200 import engine as eng_mod
from cabinet_b200 import train_engine as te
from tests import test_train_freeze_cpu as fz
from tests.test_gpu_train_variants import CASES
from tests.test_train_fp16_cpu import RecordingLib
from tests.train_variants import ARG_NAMES, ENTRY_POINTS, normalize, preconditions, variant_key

SMALL = (2, 3, 64, 96)
RUNS = [(f"{mode}-{p}", mode, c, shape, p, None) for mode, c, shape in (("large", 5, fz.SHAPE), ("small", 8, SMALL))
        for p in ("fp32", "bf16", "fp16")] + [
    ("large-bf16-all-bn-eval", "large", 5, fz.SHAPE, "bf16", fz._all_bn_eval),
    ("large-fp32-all-bn-eval", "large", 5, fz.SHAPE, "fp32", fz._all_bn_eval),
    ("large-bf16-backbone-frozen", "large", 5, fz.SHAPE, "bf16", fz._freeze_backbone),
    ("large-bf16-only-conv-out", "large", 5, fz.SHAPE, "bf16",
     lambda m: [p.requires_grad_(n == "conv_out.conv_out.weight") for n, p in m.named_parameters()])]


def record_variants(monkeypatch, mode, classes, shape, precision, freeze):
    """-> [(entry point, normalised arguments, {pointer argument: (C, ld) of the map it addresses})], and the first-write
    violations of cab_combine_backward's dg / dr."""
    # address -> (C, ld) of the map or tensor last handed out there (ld -1: a non-contiguous tensor); start-table
    # address -> the resampling operator it belongs to
    maps, tables = {}, {}
    map_ptr, tensor_ptr, tables_get = eng_mod.Map.ptr, torch.Tensor.data_ptr, te._Tables.get

    def ptr(self):
        p = map_ptr.fget(self)
        maps[p] = (self.C, self.ld)
        return p

    def data_ptr(self):
        p = tensor_ptr(self)
        maps[p] = (self.shape[-1], self.shape[-1] if self.is_contiguous() else -1)
        return p

    def get(self, kind, n_in, n_out, transpose):
        t = tables_get(self, kind, n_in, n_out, transpose)
        tables[tensor_ptr(t[0])] = (kind, n_in, n_out, transpose)
        return t

    outs = []   # (index of the next ABI call, address of the gradient view, accumulate flag)
    recs = []

    class Rec(RecordingLib):
        def __init__(self):
            super().__init__()
            self.ctx = []
            recs.append(self)

        def __getattr__(self, name):
            fn = super().__getattr__(name)

            def call(*args):
                self.ctx.append({a: maps.get(a) for a in args if isinstance(a, int) and a > 4096})
                return fn(*args)

            return call

    grads_out = te._Grads.out

    def out(self, m):
        view, acc = grads_out(self, m)
        outs.append((len(recs[-1].calls), view.ptr, view.C, acc))
        return view, acc

    monkeypatch.setattr(eng_mod.Map, "ptr", property(ptr))
    monkeypatch.setattr(torch.Tensor, "data_ptr", data_ptr)
    monkeypatch.setattr(te._Tables, "get", get)
    monkeypatch.setattr(te._Grads, "out", out)
    monkeypatch.setattr(fz, "RecordingLib", Rec)
    fz.record(monkeypatch, freeze, precision, mode, classes, shape)
    monkeypatch.undo()
    rec = recs[-1]
    calls, bad_writes = [], []
    for i, ((name, args), ctx) in enumerate(zip(rec.calls, rec.ctx)):
        entry = name[len("cabinet_"):]
        if entry not in ENTRY_POINTS:
            continue
        a = normalize(entry, args)
        if entry == "add":
            a["inplace"] = args[0] == args[4]
        if entry == "resample_sep":
            a["y_op"], a["x_op"] = tables.get(args[16]), tables.get(args[19])
        named = dict(zip(ARG_NAMES[entry], args))
        calls.append((entry, a, {k: ctx.get(v) for k, v in named.items() if isinstance(v, int) and v in ctx}))
        if entry == "cab_combine_backward":
            for k in ("dg", "dr"):
                firsts = [acc for j, p, c, acc in outs if j == i and p == named[k]]
                if not firsts or firsts[-1] != 0:
                    bad_writes.append((k, firsts))
    return calls, bad_writes


@pytest.fixture(scope="module")
def census():
    mp = pytest.MonkeyPatch()
    keys, bad_writes, calls = defaultdict(list), [], []
    try:
        for run, *args in RUNS:
            c, bw = record_variants(mp, *args)
            bad_writes += [(run, w) for w in bw]
            for entry, a, maps in c:
                keys[variant_key(entry, a)].append((run, a))
                calls.append((run, entry, a, maps))
    finally:
        mp.undo()
    return keys, calls, bad_writes


def test_every_recorded_variant_has_a_gpu_case(census):
    keys = census[0]
    matrix = {variant_key(entry, a) for entry, a in CASES}
    missing = sorted(set(keys) - matrix)
    per_entry = defaultdict(int)
    for k in keys:
        per_entry[k.split()[0]] += 1
    print(f"{len(keys)} variant keys:", dict(sorted(per_entry.items())))
    assert set(per_entry) == set(ENTRY_POINTS), set(ENTRY_POINTS) - set(per_entry)
    assert not missing, "variant keys without a case in tests/test_gpu_train_variants.py CASES:\n" + "\n".join(
        f"  {k}\n    e.g. {keys[k][0][0]}: {keys[k][0][1]}" for k in missing)


def test_gpu_cases_are_distinct_and_named_by_their_key():
    ks = [variant_key(entry, a) for entry, a in CASES]
    assert len(set(ks)) == len(ks), [k for k in ks if ks.count(k) > 1]


def test_recorded_calls_meet_the_documented_preconditions(census):
    _, calls, _ = census
    bad = []
    for run, entry, a, maps in calls:
        errs = preconditions(entry, a)
        if entry == "cab_combine_backward":   # no stride argument: dense [n_pixels][C]
            errs += [f"{k} has ld {maps[k][1]} != C {a['C']}" for k in ("g", "x", "r", "dg", "dx", "dr")
                     if maps.get(k) is None or maps[k][1] != a["C"]]
        if entry == "softmax_backward":       # dense rows of `cols`
            errs += [f"{k} is not dense [rows][{a['cols']}]: {maps.get(k)}" for k in ("p", "dp", "ds")
                     if maps.get(k) != (a["cols"], a["cols"])]
        if errs:
            bad.append((run, entry, errs))
    assert not bad, bad[:10]


def test_cab_combine_backward_outputs_are_first_writes(census):
    assert not census[2], census[2]

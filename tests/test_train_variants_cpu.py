"""CPU: the variant census of the kernels the training step launches.

The step runs against the recording double of the C-ABI (``tests/test_train_fp16_cpu.py``) for Large and Small in
fp32, bf16 and fp16, and for the freeze settings of ``tests/test_train_freeze_cpu.py``.  Every call to an entry point
of ``tests/train_variants.py`` gets its variant key (the inputs of its host dispatch).

* every ABI function the step calls is an entry point of the census (``EXEMPT`` would name the exceptions, with a
  reason), so a kernel that joins the step is counted;
* every recorded key has a case in the GPU replay matrices of ``tests/test_gpu_train_variants.py`` and
  ``tests/test_gpu_train_variants_tc.py``, so a schedule change that reaches a new kernel path fails here until that
  path is tested on the GPU;
* the documented preconditions hold: ``ld >= C`` for every strided operand, dense ``g``, ``x``, ``r``, ``dg``, ``dx``,
  ``dr`` for ``cab_combine_backward`` and dense rows for ``softmax_backward`` (their ABI has no stride);
* ``cab_combine_backward`` overwrites ``dg`` and ``dr``: the gradient regions it is given are first writes;
* the tensor-core GEMMs get what their producers made: weight packs of the GEMM's own shape, type and orientation,
  the im2col matrix's pixel stride, consistent output sizes and parity views.
"""

from collections import defaultdict

import pytest
import torch

from cabinet_b200 import engine as eng_mod
from cabinet_b200 import train_engine as te
from tests import test_train_freeze_cpu as fz
from tests.test_gpu_train_variants import CASES
from tests.test_gpu_train_variants_tc import CASES as TC_CASES
from tests.test_train_fp16_cpu import RecordingLib
from tests.train_variants import ARG_NAMES, ENTRY_POINTS, entry_of, named_args, normalize, preconditions, variant_key

SMALL = (2, 3, 64, 96)
RUNS = [(f"{mode}-{p}", mode, c, shape, p, None) for mode, c, shape in (("large", 5, fz.SHAPE), ("small", 8, SMALL))
        for p in ("fp32", "bf16", "fp16")] + [
    ("large-bf16-all-bn-eval", "large", 5, fz.SHAPE, "bf16", fz._all_bn_eval),
    ("large-fp32-all-bn-eval", "large", 5, fz.SHAPE, "fp32", fz._all_bn_eval),
    ("large-bf16-backbone-frozen", "large", 5, fz.SHAPE, "bf16", fz._freeze_backbone),
    ("large-bf16-only-conv-out", "large", 5, fz.SHAPE, "bf16",
     lambda m: [p.requires_grad_(n == "conv_out.conv_out.weight") for n, p in m.named_parameters()])]

ALL_CASES = CASES + TC_CASES
# ABI functions the step may call outside the census: (name, reason)
EXEMPT = ()


def record_variants(monkeypatch, mode, classes, shape, precision, freeze):
    """-> [(entry point, normalised arguments, {pointer argument: (C, ld) of the map it addresses}, {argument: raw value})]
    in call order (an ABI function outside the census appears as (its name, None, None, None)), and the first-write
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
        entry = entry_of(name)
        if entry is None:
            calls.append((name, None, None, None))   # outside the census: test_every_called_entry_point_is_in_the_census
            continue
        args = named_args(name, args)
        a = normalize(entry, args)
        if entry == "add":
            a["inplace"] = args[0] == args[4]
        if entry == "resample_sep":
            a["y_op"], a["x_op"] = tables.get(args[16]), tables.get(args[19])
        named = dict(zip(ARG_NAMES[entry], args))
        if entry in ("conv_tc", "conv_tc_imgw"):
            a["res_is_y"] = named["res"] is not None and named["res"] == named["y"]
            named["_dgrad"] = any(j <= i and p == named["y"] for j, p, _, _ in outs)   # writes a gradient region
        calls.append((entry, a, {k: ctx.get(v) for k, v in named.items() if isinstance(v, int) and v in ctx}, named))
        if entry == "cab_combine_backward":
            for k in ("dg", "dr"):
                firsts = [acc for j, p, c, acc in outs if j == i and p == named[k]]
                if not firsts or firsts[-1] != 0:
                    bad_writes.append((k, firsts))
    return calls, bad_writes


@pytest.fixture(scope="module")
def census():
    mp = pytest.MonkeyPatch()
    keys, bad_writes, calls, runs = defaultdict(list), [], [], {}
    try:
        for run, *args in RUNS:
            c, bw = record_variants(mp, *args)
            bad_writes += [(run, w) for w in bw]
            runs[run] = c
            for entry, a, maps, named in c:
                if a is None:
                    continue
                keys[variant_key(entry, a)].append((run, a))
                calls.append((run, entry, a, maps))
    finally:
        mp.undo()
    return keys, calls, bad_writes, runs


def test_every_called_entry_point_is_in_the_census(census):
    """Every ABI function the step calls is an entry point of the census (or exempt, with its reason), so a kernel that
    joins the step without a GPU variant case fails here."""
    exempt = {name for name, _ in EXEMPT}
    outside = defaultdict(set)
    for run, c in census[3].items():
        for entry, a, _, _ in c:
            if a is None and entry not in exempt:
                outside[entry].add(run)
    assert not outside, "entry points the step calls outside tests/train_variants.py ENTRY_POINTS:\n" + "\n".join(
        f"  {n}: {sorted(r)}" for n, r in sorted(outside.items()))


def test_every_recorded_variant_has_a_gpu_case(census):
    keys = census[0]
    matrix = {variant_key(entry, a) for entry, a in ALL_CASES}
    missing = sorted(set(keys) - matrix)
    per_entry = defaultdict(int)
    for k in keys:
        per_entry[k.split()[0]] += 1
    print(f"{len(keys)} variant keys over {len(per_entry)} entry points:", dict(sorted(per_entry.items())))
    assert set(per_entry) == set(ENTRY_POINTS), set(ENTRY_POINTS) - set(per_entry)
    assert not missing, "variant keys without a case in tests/test_gpu_train_variants*.py CASES:\n" + "\n".join(
        f"  {k}\n    e.g. {keys[k][0][0]}: {keys[k][0][1]}" for k in missing)


def test_gpu_cases_are_distinct_and_named_by_their_key():
    ks = [variant_key(entry, a) for entry, a in ALL_CASES]
    assert len(set(ks)) == len(ks), [k for k in ks if ks.count(k) > 1]


def test_recorded_calls_meet_the_documented_preconditions(census):
    _, calls, _, _ = census
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


def _c(a, b):
    return -(-a // b) * b


def test_tensor_core_operands_match_their_producers(census):
    """The conv_tc kernels trust their weight packs, the im2col matrix and the output size they are given:
    * conv_tc reads the most recent pack written at its w_packed address: pack_conv_weight with rows_pad = ceil16(Cout),
      k_pad = ceil64(Cin) per tap, the GEMM's type and taps, in the GEMM's own Cin / Cout; transpose_flip = 1 exactly for
      the data gradients (the calls of the backward, whose output is a gradient region);
    * conv_tc_view reads a pack_conv_weight_parity pack of the same (KH2, KW2, pad2), and writes the parity class
      (py, px) of the pack: hc / wc and the sub-filter agree with TrainEngine._parity_geom;
    * conv_tc_imgw reads per-image [Cout][Cin] weights (the attention's K and V^T maps): w_image_stride = Cout * Cin,
      Cin % 64 == 0;
    * a GEMM over an im2col matrix has Cin = ldx = the ld of that im2col_nchw call;
    * OH, OW of conv_tc / conv_tc_imgw are (H + 2 pad - k) / stride + 1."""
    bad = []
    for run, c in census[3].items():
        packs, cols = {}, {}
        for i, (entry, a, _, n) in enumerate(c):
            if a is None:
                continue
            if entry in ("pack_conv_weight", "pack_conv_weight_parity"):
                packs[n["out"]] = (entry, n)
            elif entry == "im2col_nchw":
                cols[n["out"]] = n
            if entry not in ("conv_tc", "conv_tc_view", "conv_tc_imgw"):
                continue
            errs = []
            Cin, Cout = n["Cin"], n["Cout"]
            if entry != "conv_tc_view":
                k_ok = all(o == (h + 2 * n["pad"] - k) // n["stride"] + 1
                           for o, h, k in ((n["OH"], n["H"], n["KH"]), (n["OW"], n["W"], n["KW"])))
                errs += [] if k_ok else [f"OH, OW {n['OH']}, {n['OW']} do not follow from H, W, k, stride, pad"]
            if n["x"] in cols:
                ld = cols[n["x"]]["ld"]
                errs += [] if Cin == ld == n["ldx"] else [f"im2col ld {ld} != Cin {Cin} / ldx {n['ldx']}"]
            if entry == "conv_tc_imgw":
                errs += [] if n["w_image_stride"] == Cout * Cin and Cin % 64 == 0 else [
                    f"w_image_stride {n['w_image_stride']} != Cout * Cin or Cin % 64"]
            else:
                pe, p = packs.get(n["w_packed"], (None, None))
                want = "pack_conv_weight" if entry == "conv_tc" else "pack_conv_weight_parity"
                if pe != want:
                    errs.append(f"w_packed was last written by {pe}, not {want}")
                else:
                    flip = p["transpose_flip"] if entry == "conv_tc" else 1
                    rows, k = (p["Cin"], p["Cout"]) if flip else (p["Cout"], p["Cin"])
                    taps = (p["KH"], p["KW"]) if entry == "conv_tc" else (p["KH2"], p["KW2"])
                    errs += [f"pack {k_} != {v}" for k_, v, w in (
                        ("rows", rows, Cout), ("k", k, Cin), ("rows_pad", p["rows_pad"], _c(Cout, 16)),
                        ("k_pad", p["k_pad"], _c(Cin, 64)), ("type", p["out_dtype"], n["op_dtype"]),
                        ("taps", taps, (n["KH"], n["KW"]))) if v != w]
                    if entry == "conv_tc" and bool(flip) != n["_dgrad"]:
                        errs.append(f"transpose_flip {flip} for a {'data-gradient' if n['_dgrad'] else 'forward'} GEMM")
                    if entry == "conv_tc_view":
                        W = n["y_sh"] // 2
                        H = n["y_sn"] // W
                        geo = [te.TrainEngine._parity_geom(p["K"], p["pad"], q) for q in (p["py"], p["px"])]
                        errs += [] if (p["pad2"], n["pad"], n["y_sw"]) == (geo[0][1], geo[0][1], 2) and \
                            (p["KH2"], p["KW2"]) == (geo[0][0], geo[1][0]) and geo[0][1] == geo[1][1] else [
                            f"sub-filter {p['KH2']}x{p['KW2']}/p{p['pad2']} != _parity_geom {geo}"]
                        errs += [] if (n["OH"], n["OW"]) == ((H - p["py"] + 1) // 2, (W - p["px"] + 1) // 2) else [
                            f"hc, wc {n['OH']}, {n['OW']} != parity ({p['py']}, {p['px']}) of {H} x {W}"]
            if errs:
                bad.append((run, i, entry, errs))
    assert not bad, bad[:10]

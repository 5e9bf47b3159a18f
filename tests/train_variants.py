"""Variant keys of the training step's elementwise and reduction kernels (``csrc/train.cu``, ``channel_sum``).

A call's variant key is what the host dispatch of its entry point looks at: the element types, whether each strided
operand is a channel window (``ld > C``), the vector-path conditions (``ld % V``, base pointer mod 16, ``C % V``,
``C / V > 256``), the shared-memory-staged "rt" threshold (``M * C >= 2^20``), ``accumulate``, ``act``, the optional
pointers that are NULL and, for ``resample_sep``, the flag bits and the channel layout.  ``tests/test_train_variants_cpu.py``
records the step's calls and checks that every key it finds has a case in ``tests/test_gpu_train_variants.py``.

A call is first normalised with :func:`normalize`: ``{argument name: value}`` from the header, with every pointer
replaced by its address mod 16 (``None`` stays ``None``) and the stream and scratch pointers dropped.
"""

import re
from pathlib import Path

HEADER = Path(__file__).resolve().parent.parent / "include" / "cabinet_b200.h"

ENTRY_POINTS = ("bn_train_stats", "bn_train_backward", "bn_frozen_backward", "affine_act", "add", "col_sum",
                "gate_scale_backward", "gate_apply_backward", "gate_mlp_backward", "cab_combine_backward",
                "softmax_backward", "conv_dgrad", "conv_wgrad", "dwconv_dgrad", "dwconv_wgrad", "resample_sep",
                "channel_sum")
DT_NAMES = {0: "f32", 1: "bf16", 2: "f16"}
RT_ROWS = 1 << 20        # rt_plan: M * C >= 2^20 elements
RED_THREADS = 256


def _arg_names():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    out = {}
    for name in ENTRY_POINTS:
        m = re.search(r"\bcabinet_%s\s*\(([^)]*)\)" % name, text)
        out[name] = [re.split(r"[\s*]+", a.strip())[-1] for a in m.group(1).split(",")]
    return out


ARG_NAMES = _arg_names()
_SKIP = {"stream", "scratch"}
# pointer arguments: the addresses whose alignment the dispatch may test, and the optional operands
_POINTERS = {
    "bn_train_stats": {"x", "gamma", "beta", "running_mean", "running_var", "stats"},
    "bn_train_backward": {"dy", "z", "stats", "dgamma", "dbeta", "dz"},
    "bn_frozen_backward": {"dy", "z", "stats", "dgamma", "dbeta", "dz"},
    "affine_act": {"z", "scale", "shift", "gate", "res", "y"},
    "add": {"a", "b", "out"},
    "col_sum": {"x", "out"},
    "gate_scale_backward": {"dy", "v", "s", "ds"},
    "gate_apply_backward": {"dy", "v", "s", "dm", "dv"},
    "gate_mlp_backward": {"mean", "w1", "w2", "hidden", "s", "ds", "dw1", "db1", "dw2", "db2", "dmean"},
    "cab_combine_backward": {"dout", "g", "x", "r", "gamma", "dg", "dx", "dr", "dgamma"},
    "softmax_backward": {"p", "dp", "ds"},
    "conv_dgrad": {"dy", "w_packed", "dx"},
    "conv_wgrad": {"dy", "x", "dw_oihw"},
    "dwconv_dgrad": {"dy", "w_packed", "dx"},
    "dwconv_wgrad": {"dy", "x", "dw"},
    "resample_sep": {"in", "out", "y_start", "y_index", "y_weight", "x_start", "x_index", "x_weight"},
    "channel_sum": {"x", "out"},
}


def normalize(entry, args):
    """(``cabinet_<entry>`` arguments) -> {name: value}, pointers as address mod 16 or None."""
    names = ARG_NAMES[entry]
    assert len(names) == len(args), (entry, len(names), len(args))
    out = {}
    for n, v in zip(names, args):
        if n in _SKIP:
            continue
        if n in _POINTERS[entry]:
            v = None if v is None else int(getattr(v, "value", v) or 0) % 16
        out[n] = v
    return out


def _win(a, ptr, ld, C, V):
    """dispatch inputs of one strided operand: window or dense, ld % V, 16-byte aligned base."""
    if a[ptr] is None:
        return f"{ptr}:null"
    return f"{ptr}:{'win' if a[ld] > C else 'dense'}{'' if a[ld] % V == 0 else '/ld%' + str(V)}" \
           f"{'' if a[ptr] == 0 else '/al' + str(a[ptr])}"


def variant_key(entry, a):
    """The variant key of one normalised call: a short string, stable across runs (it names the GPU test case)."""
    dt = DT_NAMES.get(a.get("dtype", a.get("z_dtype", a.get("in_dtype"))))
    V = 4 if dt == "f32" else 8
    parts = [entry, dt]
    if entry == "bn_train_stats":
        C = a["C"]
        parts += [_win(a, "x", "ldx", C, V), f"C%{V}={C % V}", "C/8>256" if C // 8 > RED_THREADS else "",
                  "rt" if a["M"] * C >= RT_ROWS and dt != "f32" else ""]
    elif entry in ("bn_train_backward", "bn_frozen_backward"):
        C = a["C"]
        parts += [_win(a, "dy", "lddy", C, V), _win(a, "z", "ldz", C, V), _win(a, "dz", "lddz", C, V),
                  f"C%{V}={C % V}", "C/V>256" if C // V > RED_THREADS else "",
                  "rt" if a["M"] * C >= RT_ROWS and dt != "f32" and entry == "bn_train_backward" else "",
                  f"act{a['act']}", f"acc{a['accumulate']}",
                  "dgamma:null" if a["dgamma"] is None else "", "dbeta:null" if a["dbeta"] is None else ""]
    elif entry == "affine_act":
        C = a["C"]
        parts[1] = f"{dt}>{DT_NAMES[a['y_dtype']]}"
        parts += [_win(a, "z", "ldz", C, 8), _win(a, "y", "ldy", C, 8),
                  _win(a, "res", "ldres", C, 8) if a["res"] is not None else "res:null",
                  f"C%8={C % 8}", "C>2048" if C > 2048 else "", "scale:null" if a["scale"] is None else "",
                  "gate:null" if a["gate"] is None else f"gate+{a['gate_plus']:g}", f"act{a['act']}"]
    elif entry == "add":
        C = a["C"]
        parts += [_win(a, "a", "lda", C, V), _win(a, "b", "ldb", C, V), _win(a, "out", "ldo", C, V),
                  "inplace" if a.get("inplace") else ""]
    elif entry == "col_sum":
        parts += [_win(a, "x", "ldx", a["C"], V), f"acc{a['accumulate']}"]
    elif entry == "gate_scale_backward":
        C = a["C"]
        parts += [_win(a, "dy", "lddy", C, V), _win(a, "v", "ldv", C, V), f"C%{V}={C % V}", f"act{a['act']}",
                  f"plus{a['plus']:g}"]
    elif entry == "gate_apply_backward":
        C = a["C"]
        parts += [_win(a, "dy", "lddy", C, V), _win(a, "v", "ldv", C, V), _win(a, "dv", "lddv", C, V),
                  f"C%{V}={C % V}", "C/V>256" if C // V > RED_THREADS else "", "N>65535" if a["N"] > 65535 else "",
                  "s:null" if a["s"] is None else f"plus{a['plus']:g}", "dm:null" if a["dm"] is None else "",
                  f"act{a['act']}", f"acc{a['accumulate']}"]
    elif entry == "gate_mlp_backward":
        parts = [entry, f"gate{a['gate']}", "db1:null" if a["db1"] is None else "", "db2:null" if a["db2"] is None else ""]
    elif entry == "cab_combine_backward":
        parts += ["dout:" + ("win" if a["ldo"] > a["C"] else "dense"), f"acc{a['accumulate_dx']}"]
    elif entry == "softmax_backward":
        parts = [entry]
    elif entry == "conv_dgrad":
        parts[1] = f"{dt}/w{DT_NAMES[a['w_dtype']]}"
        parts += [_win(a, "dy", "lddy", a["Cout"], V), _win(a, "dx", "lddx", a["Cin"], V),
                  f"s{a['stride']}", f"k{a['KH']}x{a['KW']}", f"acc{a['accumulate']}"]
    elif entry == "conv_wgrad":
        parts[1] = f"{dt}/x{DT_NAMES[a['x_dtype']]}"
        x_nchw = a["sxc"] != 1
        parts += [_win(a, "dy", "lddy", a["Cout"], V),
                  "x:nchw" if x_nchw else "x:" + ("win" if a["sxw"] > a["Cin"] else "dense"),
                  f"s{a['stride']}", f"k{a['KH']}x{a['KW']}"]
    elif entry == "dwconv_dgrad":
        C = a["C"]
        parts += [_win(a, "dy", "lddy", C, V), _win(a, "dx", "lddx", C, V), f"C%{V}={C % V}",
                  "" if a["w_packed"] == 0 else "w/al", f"s{a['stride']}", f"k{a['k']}", f"acc{a['accumulate']}"]
    elif entry == "dwconv_wgrad":
        C = a["C"]
        parts += [_win(a, "dy", "lddy", C, 2), _win(a, "x", "ldx", C, 2), f"C%2={C % 2}", f"s{a['stride']}",
                  f"k{a['k']}", "OW<8" if a["OW"] < 8 else ""]
    elif entry == "resample_sep":
        parts[1] = f"{dt}>{DT_NAMES[a['out_dtype']]}"
        flags = a["accumulate"]
        vec8 = all(a[k] % 8 == 0 for k in ("isn", "isy", "isx", "osn", "osy", "osx")) and a["C"] % 8 == 0 and \
            a["in"] == 0 and a["out"] == 0
        parts += [f"flags{flags}", "in:" + ("nhwc" if a["isc"] == 1 else "planar"),
                  "out:" + ("nhwc" if a["osc"] == 1 else "planar"),
                  "" if a["isc"] != 1 or a["isx"] == a["C"] else "in:win",
                  "" if a["osc"] != 1 or a["osx"] == a["C"] else "out:win",
                  "v8" if vec8 else ""]
    elif entry == "channel_sum":
        parts += [_win(a, "x", "ldx", a["C"], V)]
    else:
        raise KeyError(entry)
    return " ".join(p for p in parts if p)


def preconditions(entry, a):
    """Documented preconditions of one normalised call that the kernels do not check: a list of violations."""
    bad = []
    for ptr, ld, C in _STRIDED.get(entry, ()):
        if a.get(ptr) is not None and a[ld] < a[C]:
            bad.append(f"{ld}={a[ld]} < {C}={a[C]}")
    return bad


# (pointer, its pixel stride, its channel count) of every strided operand
_STRIDED = {
    "bn_train_stats": [("x", "ldx", "C")],
    "bn_train_backward": [("dy", "lddy", "C"), ("z", "ldz", "C"), ("dz", "lddz", "C")],
    "bn_frozen_backward": [("dy", "lddy", "C"), ("z", "ldz", "C"), ("dz", "lddz", "C")],
    "affine_act": [("z", "ldz", "C"), ("res", "ldres", "C"), ("y", "ldy", "C")],
    "add": [("a", "lda", "C"), ("b", "ldb", "C"), ("out", "ldo", "C")],
    "col_sum": [("x", "ldx", "C")],
    "gate_scale_backward": [("dy", "lddy", "C"), ("v", "ldv", "C")],
    "gate_apply_backward": [("dy", "lddy", "C"), ("v", "ldv", "C"), ("dv", "lddv", "C")],
    "cab_combine_backward": [("dout", "ldo", "C")],
    "conv_dgrad": [("dy", "lddy", "Cout"), ("dx", "lddx", "Cin")],
    "conv_wgrad": [("dy", "lddy", "Cout")],
    "dwconv_dgrad": [("dy", "lddy", "C"), ("dx", "lddx", "C")],
    "dwconv_wgrad": [("dy", "lddy", "C"), ("x", "ldx", "C")],
    "channel_sum": [("x", "ldx", "C")],
}

"""Variant keys of the kernels the training step launches.

A call's variant key is what the host dispatch of its entry point looks at.  For the elementwise and reduction kernels
(``csrc/train.cu``, ``channel_sum``) these are the element types, whether each strided operand is a channel window
(``ld > C``), the vector-path conditions (``ld % V``, base pointer mod 16, ``C % V``, ``C / V > 256``), the
shared-memory-staged "rt" threshold (``M * C >= 2^20``), ``accumulate``, ``act``, the optional pointers that are NULL and,
for ``resample_sep``, the flag bits and the channel layout.  For the tensor-core convolutions (``conv_tc_impl``,
``wg_plan``, ``cabinet_dwconv_tma_dt``) they are the plan the host derives from the shapes: flat or tiled walk, the
TW x TH patch and whether the output leaves a tail, ragged K blocks, several N / M tiles, resident weights, the finalize
kernel, the channel chunks.  ``tests/test_train_variants_cpu.py`` records the step's calls and checks that every key it
finds has a case in ``tests/test_gpu_train_variants.py`` or ``tests/test_gpu_train_variants_tc.py``.

A call is first normalised with :func:`normalize`: ``{argument name: value}`` from the header, with every pointer
replaced by its address mod 16 (``None`` stays ``None``) and the stream and scratch pointers dropped.  ``cabinet_X`` of
an entry point with a ``cabinet_X_dt`` variant is ``cabinet_X_dt(..., CABINET_BF16)``: both normalise to the entry ``X``
with the operand type as an argument (:func:`named_args`).
"""

import re
from pathlib import Path

HEADER = Path(__file__).resolve().parent.parent / "include" / "cabinet_b200.h"

ENTRY_POINTS = ("bn_train_stats", "bn_train_backward", "bn_frozen_backward", "affine_act", "add", "col_sum",
                "gate_scale_backward", "gate_apply_backward", "gate_mlp_backward", "cab_combine_backward",
                "softmax_backward", "conv_dgrad", "conv_wgrad", "dwconv_dgrad", "dwconv_wgrad", "resample_sep",
                "channel_sum",
                # tensor-core convolutions
                "conv_tc", "conv_tc_view", "conv_tc_imgw", "conv_wgrad_tc", "conv_wgrad_tc_batched", "dwconv_tma",
                # weight packers and layout helpers
                "pack_conv_weight", "pack_conv_weight_parity", "pack_dw_weight", "embed_filter", "im2col_nchw",
                "transpose_tokens",
                # attention softmax
                "attn_softmax", "attn_softmax_backward",
                # CUDA-core forward kernels
                "conv2d_simt", "dwconv", "gate_fc", "cab_combine", "softmax_rows", "upsample_logits_nchw",
                # eval-mode BatchNorm
                "bn_frozen_stats")
# entry points whose cabinet_X is cabinet_X_dt(..., CABINET_BF16): the census reads the _dt prototype
DT_ENTRIES = ("conv_tc", "conv_tc_view", "conv_tc_imgw", "conv_wgrad_tc", "conv_wgrad_tc_batched", "dwconv_tma",
              "im2col_nchw", "pack_conv_weight_parity", "attn_softmax", "attn_softmax_backward", "transpose_tokens")
DT_NAMES = {0: "f32", 1: "bf16", 2: "f16"}
RT_ROWS = 1 << 20        # rt_plan: M * C >= 2^20 elements
RED_THREADS = 256
SMS = 148                # wg_plan sizes its pixel splits for 148 SMs


def _prototypes():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    names, pointers = {}, {}
    for name in ENTRY_POINTS:
        m = re.search(r"\bcabinet_%s%s\s*\(([^)]*)\)" % (name, "_dt" if name in DT_ENTRIES else ""), text)
        args = [a.strip() for a in m.group(1).split(",")]
        names[name] = [re.split(r"[\s*]+", a)[-1] for a in args]
        pointers[name] = {n for a, n in zip(args, names[name]) if "*" in a}
    return names, pointers


# argument names of every entry point, and the pointer arguments among them (the addresses whose alignment a dispatch
# may test, and the optional operands)
ARG_NAMES, _POINTERS = _prototypes()
_SKIP = {"stream", "scratch"}


def entry_of(name):
    """ABI function name -> its census entry point (``cabinet_X_dt`` -> ``X``), or None."""
    e = name[len("cabinet_"):]
    if e.endswith("_dt") and e[:-3] in DT_ENTRIES:
        return e[:-3]
    return e if e in ENTRY_POINTS else None


def named_args(name, args):
    """The argument list of a recorded ``cabinet_X`` / ``cabinet_X_dt`` call in the order of ``ARG_NAMES[X]``."""
    entry = entry_of(name)
    args = list(args)
    if entry in DT_ENTRIES and not name.endswith("_dt"):
        args = args[:-1] + [1] + args[-1:]   # cabinet_X(...) = cabinet_X_dt(..., CABINET_BF16, stream)
    assert len(ARG_NAMES[entry]) == len(args), (name, len(ARG_NAMES[entry]), len(args))
    return args


def normalize(entry, args):
    """(arguments in the order of ``ARG_NAMES[entry]``) -> {name: value}, pointers as address mod 16 or None."""
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
    elif entry in _NEW_KEYS:
        parts = _NEW_KEYS[entry](entry, a)
    else:
        raise KeyError(entry)
    return " ".join(p for p in parts if p)


def _cdiv(a, b):
    return -(-a // b)


def _patch(OW, OH, M):
    """The TH x TW = M patch with the least covered area, ties to the wider one (conv_tc_impl / wg_plan)."""
    best = None
    tw = M
    while tw >= (4 if M == 128 else 2):
        th = M // tw
        cover = _cdiv(OW, tw) * tw * _cdiv(OH, th) * th
        if best is None or cover < best[0]:
            best = (cover, tw, th)
        tw //= 2
    return best[1], best[2]


def tc_plan(entry, a):
    """The host plan of conv_tc_impl for a conv_tc / conv_tc_view / conv_tc_imgw call."""
    view = entry == "conv_tc_view"
    stride = 1 if view else a["stride"]
    KH, KW, Cin, Cout = a["KH"], a["KW"], a["Cin"], a["Cout"]
    flat = KH == 1 and KW == 1 and stride == 1 and a["pad"] == 0 and not view
    nkb = KH * KW * _cdiv(Cin, 64)
    n16 = _cdiv(Cout, 16) * 16
    n_tiles = _cdiv(n16, 256)
    block_n = n16 if n_tiles == 1 else 256
    y_dtype = a["op_dtype"] if view else a["y_dtype"]
    per_image = entry == "conv_tc_imgw"
    if flat:
        P = a["N"] * a["H"] * a["W"]
        TW, TH, OW, OH = 128, 1, P, 1
    else:
        OW, OH = a["OW"], a["OH"]
        TW, TH = _patch(OW, OH, 128)
    return dict(flat=flat, stride=stride, n_tiles=n_tiles, block_n=block_n, y_dtype=y_dtype, TW=TW, TH=TH, OW=OW, OH=OH,
                b_resident=not per_image and n_tiles == 1 and nkb * block_n * 64 * 2 <= 80 * 1024,
                c_bufs=2 if y_dtype != 0 and block_n > 64 else 1)


def _tc_key(entry, a):
    g = tc_plan(entry, a)
    Cin, Cout = a["Cin"], a["Cout"]
    parts = [entry, f"{DT_NAMES[a['op_dtype']]}>{DT_NAMES[g['y_dtype']]}"]
    if g["flat"]:
        parts.append("flat" + ("/P%128" if g["OW"] % 128 else ""))
    else:
        parts += [f"s{g['stride']} k{a['KH']}x{a['KW']}", f"{g['TW']}x{g['TH']}" + ("/owtail" if g["OW"] % g["TW"] else "")
                  + ("/ohtail" if g["OH"] % g["TH"] else "")]
    if entry == "conv_tc_view":
        parts.append(f"view/p{a['pad']}")
    parts += ["cin<64" if Cin < 64 else ("cin%64" if Cin % 64 else ""), "ntiles>1" if g["n_tiles"] > 1 else "",
              "cout%64" if Cout % 64 else "", "bres" if g["b_resident"] else "", f"cbufs{g['c_bufs']}",
              "x:win" if a["ldx"] > Cin else "", "y:win" if a["ldy"] > Cout else ""]
    if entry != "conv_tc_view":
        parts += ["" if a["res"] is None else ("res=y" if a.get("res_is_y") else "res"), f"act{a['act']}" if a["act"] else ""]
    return parts


def wg_plan(a, per_image=False):
    """The host plan of wgrad_tc_impl (wg_plan, the finalize choice) for a conv_wgrad_tc / _batched call."""
    N, H, W, Cin, Cout = a["N"], a["H"], a["W"], a["Cin"], a["Cout"]
    KH, stride, pad = (1, 1, 0) if per_image else (a["KH"], a["stride"], a["pad"])
    OH, OW = (H + 2 * pad - KH) // stride + 1, (W + 2 * pad - KH) // stride + 1
    flat = KH == 1 and stride == 1
    if flat:
        TW, TH, n_k_tiles = 64, 1, _cdiv(N * OH * OW, 64)
    else:
        TW, TH = _patch(OW, OH, 64)
        n_k_tiles = N * _cdiv(OW, TW) * _cdiv(OH, TH)
    NB = 64 if Cin <= 64 else (128 if Cin <= 128 else 256)
    n_tiles, m_tiles = _cdiv(Cin, NB), _cdiv(Cout, 128)
    base = m_tiles * n_tiles * KH * KH
    splits = min(max(1, min((SMS * (2 if NB <= 128 else 1)) // base, n_k_tiles)), 1024)
    tps = _cdiv(n_k_tiles, splits)
    splits = N if per_image else _cdiv(n_k_tiles, tps)
    total = Cout * Cin * KH * KH
    fin = "none" if per_image else ("par" if splits >= 64 or (splits >= 16 and total <= 65536) else "seq")
    return dict(flat=flat, OH=OH, OW=OW, TW=TW, TH=TH, NB=NB, n_tiles=n_tiles, m_tiles=m_tiles, splits=splits, fin=fin,
                stride=stride, KH=KH)


def _wg_key(entry, a):
    g = wg_plan(a, entry == "conv_wgrad_tc_batched")
    Cin, Cout = a["Cin"], a["Cout"]
    parts = [entry, DT_NAMES[a["op_dtype"]]]
    if entry == "conv_wgrad_tc":
        if g["flat"]:
            parts.append("flat" + ("/P%64" if (a["N"] * a["H"] * a["W"]) % 64 else ""))
        else:
            parts += [f"s{g['stride']} k{g['KH']}", f"{g['TW']}x{g['TH']}" + ("/owtail" if g["OW"] % g["TW"] else "")
                      + ("/ohtail" if g["OH"] % g["TH"] else ""),
                      "oddH" if g["stride"] == 2 and a["H"] % 2 else "", "oddW" if g["stride"] == 2 and a["W"] % 2 else ""]
        parts.append(f"fin:{g['fin']}")
    ld_dy = a["lddy"] if entry == "conv_wgrad_tc" else a["lda"]
    parts += [f"NB{g['NB']}", "ntiles>1" if g["n_tiles"] > 1 else "", "mtiles>1" if g["m_tiles"] > 1 else "",
              "cin%64" if Cin % 64 else "", "cout%128" if Cout % 128 else "",
              "dy:win" if ld_dy > Cout else "", "x:win" if a["ldx"] > Cin else ""]
    return parts


def dw_chunks(C):
    """Channel widths of the balanced chunks of cabinet_dwconv_tma_dt."""
    n = _cdiv(C, 64)
    CB = _cdiv(_cdiv(C, n), 8) * 8
    return sorted({min(CB, C - i * CB) for i in range(n)})


def _dwtma_key(entry, a):
    C = a["C"]
    return [entry, DT_NAMES[a["op_dtype"]], f"k{a['k']} s{a['stride']}", "cw" + "/".join(map(str, dw_chunks(C))),
            "x:win" if a["ldx"] > C else "", "y:win" if a["ldy"] > C else "", "ow%16" if a["OW"] % 16 else "",
            "oh%8" if a["OH"] % 8 else "", f"act{a['act']}" if a["act"] else "", "" if a["gap_sum"] is None else "gap"]


def _pack_key(entry, a):
    if entry == "pack_conv_weight":
        flip = a["transpose_flip"]
        rows, k = (a["Cin"], a["Cout"]) if flip else (a["Cout"], a["Cin"])
        return [entry, DT_NAMES[a["out_dtype"]], f"flip{flip}", f"k{a['KH']}x{a['KW']}",
                "rowpad" if a["rows_pad"] > rows else "", "kpad" if a["k_pad"] > k else ""]
    if entry == "pack_conv_weight_parity":
        return [entry, DT_NAMES[a["out_dtype"]], f"k{a['K']}/p{a['pad']} py{a['py']}px{a['px']}",
                f"{a['KH2']}x{a['KW2']}/p{a['pad2']}", "rowpad" if a["rows_pad"] > a["Cin"] else "",
                "kpad" if a["k_pad"] > a["Cout"] else ""]
    if entry == "pack_dw_weight":
        return [entry, f"k{a['k']}", f"flip{a['flip']}"]
    return [entry, f"k{a['k']}>K{a['K']}", "extract_add" if a["extract_add"] else "embed"]   # embed_filter


IM2COL_PX = 64


def im2col_plan(a):
    """(OH, OW, row-segment kernel?) of cabinet_im2col_nchw_dt."""
    k, s, p = a["k"], a["stride"], a["pad"]
    OH, OW = (a["H"] + 2 * p - k) // s + 1, (a["W"] + 2 * p - k) // s + 1
    smem = (a["Cin"] * k * (IM2COL_PX * s + k - s) + a["ld"]) * 4
    return OH, OW, smem <= 48 * 1024 and a["N"] * OH * _cdiv(OW, IM2COL_PX) < 2 ** 31


def _layout_key(entry, a):
    if entry == "im2col_nchw":
        OH, OW, row = im2col_plan(a)
        return [entry, DT_NAMES[a["out_dtype"]], f"k{a['k']} s{a['stride']}", "row" if row else "elem",
                "segtail" if row and OW % IM2COL_PX else "", "ldpad" if a["ld"] > a["Cin"] * a["k"] ** 2 else ""]
    if entry == "transpose_tokens":
        return [entry, DT_NAMES[a["op_dtype"]], "L%32" if a["L"] % 32 else "", "C%32" if a["C"] % 32 else "",
                "x:win" if a["ldx"] > a["C"] else ""]
    # attn_softmax, attn_softmax_backward, softmax_rows
    dt = DT_NAMES[a["p_dtype"] if entry == "softmax_rows" else a["op_dtype"]]
    return [entry, dt, "cols%32" if a["cols"] % 32 else ""]


def _fwd_key(entry, a):
    if entry == "conv2d_simt":
        x = "x:nhwc" + ("/win" if a["sxw"] > a["Cin"] else "") if a["sxc"] == 1 else "x:planar"
        return [entry, f"{DT_NAMES[a['x_dtype']]}/{DT_NAMES[a['w_dtype']]}>{DT_NAMES[a['y_dtype']]}",
                "batched" if a["batches"] > 1 else "", x, "w:kfast" if a["w_sk"] == 1 else "w:cofast",
                f"s{a['stride']} k{a['KH']}x{a['KW']}", "bias:null" if a["bias"] is None else "",
                "res" if a["res"] is not None else "", "alpha" if a["alpha"] != 1 else "",
                "y:win" if a["ldy"] > a["Cout"] else "", f"act{a['act']}" if a["act"] else ""]
    if entry == "dwconv":
        C = a["C"]
        return [entry, DT_NAMES[a["dtype"]], f"k{a['k']} s{a['stride']}", "x:win" if a["ldx"] > C else "",
                "y:win" if a["ldy"] > C else "", f"act{a['act']}" if a["act"] else "", "" if a["gap_sum"] is None else "gap"]
    if entry == "gate_fc":
        vec = not a["in_fixed"] and a["C"] % 4 == 0 and a["in"] == 0
        return [entry, f"act{a['act']}", "b:null" if a["b"] is None else "", "fixed" if a["in_fixed"] else "",
                "vec" if vec else "", "N>8" if a["N"] > 8 else ""]
    if entry == "cab_combine":
        return [entry, DT_NAMES[a["dtype"]], "out:win" if a["ldo"] > a["C"] else ""]
    if entry == "upsample_logits_nchw":
        return [entry, DT_NAMES[a["y_dtype"]], "x8" if (a["OH"], a["OW"]) == (8 * a["IH"], 8 * a["IW"]) else ""]
    return [entry, "gamma:null" if a["gamma"] is None else "", "beta:null" if a["beta"] is None else ""]  # bn_frozen_stats


_NEW_KEYS = {**dict.fromkeys(("conv_tc", "conv_tc_view", "conv_tc_imgw"), _tc_key),
             **dict.fromkeys(("conv_wgrad_tc", "conv_wgrad_tc_batched"), _wg_key), "dwconv_tma": _dwtma_key,
             **dict.fromkeys(("pack_conv_weight", "pack_conv_weight_parity", "pack_dw_weight", "embed_filter"), _pack_key),
             **dict.fromkeys(("im2col_nchw", "transpose_tokens", "attn_softmax", "attn_softmax_backward", "softmax_rows"),
                             _layout_key),
             **dict.fromkeys(("conv2d_simt", "dwconv", "gate_fc", "cab_combine", "upsample_logits_nchw", "bn_frozen_stats"),
                             _fwd_key)}


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

"""ctypes binding of ``libcabinet_b200.so`` (the C-ABI declared in ``include/cabinet_b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C cabinet_b200/csrc``.  There is
no fallback: if it is missing, importing the engine raises.
"""

from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libcabinet_b200.so"
CSRC = PKG / "csrc"

F32, BF16, F16 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_HSWISH, ACT_HSIGMOID, ACT_SIGMOID = 0, 1, 2, 3, 4

_p, _i, _ll, _f = C.c_void_p, C.c_int, C.c_longlong, C.c_float

# name -> argtypes; must list every symbol include/cabinet_b200.h declares (tests/test_abi.py checks this)
SIGNATURES = {
    "cabinet_last_error": ([], C.c_char_p),
    "cabinet_abi_version": ([], _i),
    "cabinet_device_info": ([C.POINTER(_i)] * 3, _i),
    "cabinet_debug_flags": ([_i], _i),
    "cabinet_debug_read": ([_p, _i], _i),
    "cabinet_conv2d_simt": ([_p, _i, _ll, _ll, _ll, _ll, _ll, _p, _i, _ll, _ll, _ll, _p, _p, _ll, _p, _i, _ll, _ll,
                             _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _p], _i),
    "cabinet_conv_tc": ([_p, _ll, _i, _i, _i, _i, _p, _i, _i, _i, _i, _i, _p, _p, _ll, _p, _i, _ll, _i, _i, _i, _p], _i),
    "cabinet_conv_tc_dt": ([_p, _ll, _i, _i, _i, _i, _p, _i, _i, _i, _i, _i, _p, _p, _ll, _p, _i, _ll, _i, _i, _i, _i, _p],
                           _i),
    "cabinet_conv_tc_view": ([_p, _ll, _i, _i, _i, _i, _p, _i, _i, _i, _i, _p, _p, _ll, _i, _i, _ll, _ll, _ll, _p], _i),
    "cabinet_conv_tc_view_dt": ([_p, _ll, _i, _i, _i, _i, _p, _i, _i, _i, _i, _p, _p, _ll, _i, _i, _ll, _ll, _ll, _i, _p], _i),
    "cabinet_conv_tc_se": ([_p, _ll, _i, _i, _i, _i, _p, _i, _p, _i, _i, _i, _i, _i, _p, _p, _ll, _p, _i, _ll, _i, _i, _i,
                            _p], _i),
    "cabinet_conv_tc_split_act": ([_p, _ll, _i, _i, _i, _i, _p, _i, _i, _i, _i, _i, _p, _p, _i, _ll, _i, _i, _i, _i, _p], _i),
    "cabinet_conv_tc_imgw": ([_p, _ll, _i, _i, _i, _i, _p, _ll, _i, _i, _i, _i, _i, _p, _p, _ll, _p, _i, _ll, _i, _i, _i,
                              _p], _i),
    "cabinet_conv_tc_imgw_dt": ([_p, _ll, _i, _i, _i, _i, _p, _ll, _i, _i, _i, _i, _i, _p, _p, _ll, _p, _i, _ll, _i, _i, _i,
                                 _i, _p], _i),
    "cabinet_conv_tc_up": ([_p, _ll, _i, _i, _i, _i, _p, _i, _i, _i, _i, _i, _p, _p, _i, _i, _p, _ll, _i, _i, _i, _p], _i),
    "cabinet_gate_scale_weights": ([_p, _i, _f, _p, _p, _p, _p, _i, _i, _i, _p, _p, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_scale_weights": ([_p, _p, _p, _i, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_stem_tc": ([_p, _i, _i, _i, _p, _p, _p, _ll, _p, _ll, _i, _i, _p], _i),
    "cabinet_stem_tc2": ([_p, _i, _i, _i, _p, _p, _ll, _p, _ll, _i, _i, _p], _i),
    "cabinet_dwconv": ([_p, _ll, _p, _p, _p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p], _i),
    "cabinet_dwconv_tma": ([_p, _ll, _p, _p, _p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p], _i),
    "cabinet_dwconv_tma_dt": ([_p, _ll, _p, _p, _p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p], _i),
    "cabinet_mbconv_noexpand_fused": ([_p, _ll, _p, _p, _p, _p, _p, _ll, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_mbconv_fused": ([_p, _ll, _i, _i, _i, _i, _p, _p, _i, _i, _i, _i, _i, _p, _p, _i, _i, _p, _ll, _i, _i, _p,
                              _p], _i),
    "cabinet_mbconv_t": ([_p, _ll, _i, _i, _i, _i, _p, _p, _i, _i, _i, _i, _i, _p, _p, _i, _i, _p, _ll, _i, _i, _p, _p,
                          _p], _i),
    "cabinet_expand_sums": ([_p, _ll, _i, _i, _i, _i, _p, _p, _i, _i, _i, _i, _p, _p], _i),
    "cabinet_gate_mlp": ([_p, _f, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p], _i),
    "cabinet_gate_fc": ([_p, _f, _p, _p, _p, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_scale_act": ([_p, _ll, _i, _p, _i, _ll, _i, _i, _i, _p], _i),
    "cabinet_psp_pool": ([_p, _ll, _i, _p, _i, _i, _i, _i, _p, _ll, _p], _i),
    "cabinet_psp_concat": ([_p, _ll, _p, _p, _ll, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_softmax_rows": ([_p, _p, _i, _ll, _i, _p], _i),
    "cabinet_attention_tc": ([_p, _ll, _p, _ll, _p, _ll, _p, _p, _ll, _i, _i, _i, _f, _p], _i),
    "cabinet_cab_combine": ([_p, _p, _p, _p, _ll, _p, _i, _ll, _i, _p], _i),
    "cabinet_channel_sum": ([_p, _ll, _i, _i, _ll, _i, _p, _p, _ll, _p], _i),
    "cabinet_bilinear_nhwc": ([_p, _ll, _i, _p, _ll, _i, _i, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_upsample_logits_nchw": ([_p, _i, _i, _i, _i, _p, _i, _i, _i, _p], _i),
    "cabinet_upsample_argmax": ([_p, _i, _i, _i, _i, _p, _i, _i, _p, _i, _i, _p, _p], _i),
    "cabinet_normalize_u8": ([_p, _p, _i, _i, _i, _f, _f, _f, _f, _f, _f, _p], _i),
    "cabinet_confusion_hist": ([_p, _i, _p, _i, _ll, _i, _i, _p, _p], _i),
    "cabinet_upsample_softmax_accum": ([_p, _p, _i, _i, _i, _i, _i, _i, _p, _ll, _ll, _ll, _i, _i, _i, _i, _p, _p, _f,
                                        _p], _i),
    "cabinet_prob_resize_accum": ([_p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _i, _p], _i),
    "cabinet_argmax_hist_nchw": ([_p, _i, _i, _ll, _p, _p, _i, _i, _p, _p], _i),
    "cabinet_ohem_workspace_bytes": ([], _ll),
    "cabinet_train_scratch_floats": ([_ll, _i, _i], _ll),
    "cabinet_pack_conv_weight": ([_p, _i, _i, _i, _i, _p, _i, _i, _i, _i, _p], _i),
    "cabinet_pack_conv_weight_parity": ([_p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _i, _p], _i),
    "cabinet_pack_conv_weight_parity_dt": ([_p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _i, _i, _p], _i),
    "cabinet_pack_dw_weight": ([_p, _i, _i, _i, _p, _p], _i),
    "cabinet_im2col_nchw": ([_p, _i, _i, _i, _i, _i, _i, _i, _p, _ll, _p], _i),
    "cabinet_im2col_nchw_dt": ([_p, _i, _i, _i, _i, _i, _i, _i, _p, _ll, _i, _p], _i),
    "cabinet_embed_filter": ([_p, _i, _i, _i, _i, _p, _ll, _i, _p], _i),
    "cabinet_bn_train_stats": ([_p, _ll, _i, _ll, _i, _p, _p, _f, _f, _p, _p, _p, _p, _p], _i),
    "cabinet_affine_act": ([_p, _ll, _i, _p, _p, _p, _f, _p, _ll, _p, _ll, _i, _ll, _ll, _i, _i, _p], _i),
    "cabinet_bn_train_backward": ([_p, _ll, _p, _ll, _i, _p, _i, _p, _p, _p, _ll, _ll, _i, _i, _p, _p], _i),
    "cabinet_bn_frozen_stats": ([_p, _p, _p, _p, _f, _i, _p, _p], _i),
    "cabinet_bn_frozen_backward": ([_p, _ll, _p, _ll, _i, _p, _i, _p, _p, _p, _ll, _ll, _i, _i, _p, _p], _i),
    "cabinet_stem_dgrad": ([_p, _ll, _p, _ll, _i, _p, _p, _p, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_gate_scale_backward": ([_p, _ll, _p, _ll, _i, _p, _f, _i, _p, _i, _ll, _i, _p, _p], _i),
    "cabinet_gate_apply_backward": ([_p, _ll, _p, _ll, _i, _p, _f, _p, _f, _i, _p, _ll, _i, _ll, _i, _i, _p], _i),
    "cabinet_gate_mlp_backward": ([_p, _f, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p], _i),
    "cabinet_col_sum": ([_p, _ll, _i, _ll, _i, _p, _i, _p, _p], _i),
    "cabinet_conv_dgrad": ([_p, _ll, _i, _p, _i, _ll, _ll, _p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_conv_wgrad_scratch_floats": ([_i, _i, _i, _i, _i, _i, _i], _ll),
    "cabinet_conv_wgrad": ([_p, _ll, _i, _p, _i, _ll, _ll, _ll, _ll, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p,
                            _p], _i),
    "cabinet_conv_wgrad_tc_scratch_floats": ([_i, _i, _i, _i, _i, _i, _i, _i, _i], _ll),
    "cabinet_conv_wgrad_tc": ([_p, _ll, _p, _ll, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p], _i),
    "cabinet_conv_wgrad_tc_dt": ([_p, _ll, _p, _ll, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p], _i),
    "cabinet_conv_wgrad_tc_batched": ([_p, _ll, _p, _ll, _p, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_conv_wgrad_tc_batched_dt": ([_p, _ll, _p, _ll, _p, _i, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_dwconv_dgrad": ([_p, _ll, _i, _p, _p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p], _i),
    "cabinet_dwconv_wgrad": ([_p, _ll, _p, _ll, _i, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p], _i),
    "cabinet_resample_sep": ([_p, _i, _ll, _ll, _ll, _ll, _p, _i, _ll, _ll, _ll, _ll, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p,
                              _i, _p], _i),
    "cabinet_softmax_backward": ([_p, _p, _p, _ll, _i, _f, _p], _i),
    "cabinet_attn_softmax": ([_p, _f, _p, _p, _ll, _i, _p], _i),
    "cabinet_attn_softmax_dt": ([_p, _f, _p, _p, _ll, _i, _i, _p], _i),
    "cabinet_attn_softmax_backward": ([_p, _p, _p, _ll, _i, _f, _p], _i),
    "cabinet_attn_softmax_backward_dt": ([_p, _p, _p, _ll, _i, _f, _i, _p], _i),
    "cabinet_transpose_tokens": ([_p, _ll, _p, _i, _i, _i, _p], _i),
    "cabinet_transpose_tokens_dt": ([_p, _ll, _p, _i, _i, _i, _i, _p], _i),
    "cabinet_cab_combine_backward": ([_p, _ll, _p, _p, _p, _p, _i, _p, _p, _p, _p, _ll, _i, _i, _p, _p], _i),
    "cabinet_add": ([_p, _ll, _p, _ll, _p, _ll, _i, _ll, _i, _p], _i),
    "cabinet_ohem_ce_forward": ([_p, _i, _p, _i, _i, _i, _ll, _p, _i, _f, _ll, _p, _p, _p, _p], _i),
    "cabinet_ohem_ce_backward": ([_p, _i, _p, _i, _i, _i, _ll, _p, _p, _p, _p, _p, _p], _i),
}

_lib = None


def build(verbose: bool = False) -> Path:
    """Compile the library for sm_100a (nvcc cross-compiles; no GPU needed)."""
    r = subprocess.run(["make", "-C", str(CSRC), "-j8"], capture_output=True, text=True)
    if r.returncode != 0 or verbose:
        print(r.stdout[-4000:], r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building libcabinet_b200.so failed")
    return LIB_PATH


def load():
    """dlopen the library and set prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.is_file():
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(or `make -C cabinet_b200/csrc`). cabinet_b200 has no fallback path.")
        lib = C.CDLL(str(LIB_PATH))
        for name, (args, res) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = res
        _lib = lib
    return _lib


class CabinetError(RuntimeError):
    pass


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().cabinet_last_error().decode(errors="replace")
        if rc == 1:
            raise ValueError(f"{what}: {msg}")
        raise CabinetError(f"{what}: {msg}")

"""CPU: the fp16 training mode without a GPU.

* the fp16 schedule, forward and backward tape, against a recording double of the C-ABI: no bf16 operand anywhere, the
  tensor-core / staging calls are their ``*_dt`` variants with fp16, and the call counts equal the bf16 schedule's;
* entry points that do not implement fp16 reject it (return 1 with a message) before they touch a pointer;
* the compiled library has tensor-core MMAs (UTCHMMA) in the fp16 instantiations of conv_tc and conv_wgrad_tc.
"""

import ctypes
import re
import shutil
import subprocess
from collections import Counter
from pathlib import Path

import pytest
import torch

from cabinet_b200 import _lib
from cabinet_b200.synthetic import build_model

HEADER = Path(__file__).resolve().parent.parent / "include" / "cabinet_b200.h"
TC_NAMES = {"cabinet_conv_tc", "cabinet_conv_tc_view", "cabinet_conv_tc_imgw", "cabinet_conv_wgrad_tc",
            "cabinet_conv_wgrad_tc_batched", "cabinet_dwconv_tma", "cabinet_im2col_nchw", "cabinet_transpose_tokens",
            "cabinet_pack_conv_weight_parity", "cabinet_attn_softmax", "cabinet_attn_softmax_backward"}
# the entry points that implement fp16 (the ones the fp16 training schedule may pass it to)
F16_ENTRY_POINTS = {n + "_dt" for n in TC_NAMES} | {
    "cabinet_pack_conv_weight", "cabinet_conv2d_simt", "cabinet_resample_sep", "cabinet_add", "cabinet_channel_sum",
    "cabinet_bn_train_stats", "cabinet_affine_act", "cabinet_bn_train_backward", "cabinet_gate_scale_backward",
    "cabinet_gate_apply_backward", "cabinet_col_sum", "cabinet_conv_dgrad", "cabinet_conv_wgrad", "cabinet_dwconv_dgrad",
    "cabinet_dwconv_wgrad", "cabinet_cab_combine", "cabinet_cab_combine_backward"}


def dtype_positions():
    """{entry point: indices of its element-type arguments} from the header's parameter names."""
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    out = {}
    for m in re.finditer(r"(?:const\s+char\s*\*|long\s+long|int)\s+(cabinet_\w+)\s*\(([^)]*)\)\s*;", text):
        args = [a.strip() for a in m.group(2).split(",")] if m.group(2).strip() not in ("", "void") else []
        out[m.group(1)] = [i for i, a in enumerate(args)
                           if re.fullmatch(r"int\s+(\w+_)?dtype", a) and "label" not in a and "pred" not in a]
    return out


class RecordingLib:
    def __init__(self):
        self.calls = []

    def cabinet_train_scratch_floats(self, *a):
        return 16

    cabinet_conv_wgrad_scratch_floats = cabinet_conv_wgrad_tc_scratch_floats = cabinet_train_scratch_floats

    def __getattr__(self, name):
        if name not in _lib.SIGNATURES:
            raise AttributeError(name)
        argtypes, _ = _lib.SIGNATURES[name]

        def fn(*args):
            assert len(args) == len(argtypes), f"{name}: {len(args)} args, ABI has {len(argtypes)}"
            for a, t in zip(args, argtypes):
                t.from_param(a) if hasattr(t, "from_param") else t(a)
            self.calls.append((name, args))
            return 0

        return fn


def record_step(monkeypatch, mode, C, shape, precision):
    from cabinet_b200 import train_engine as te

    rec = RecordingLib()
    monkeypatch.setattr(_lib, "load", lambda: rec)
    monkeypatch.setattr(te.TrainEngine, "stream", property(lambda self: None))
    model = build_model(C, mode).train()

    class P:
        is_cuda = True
        device = torch.device("cpu")

    real_next = next
    monkeypatch.setattr(te, "next", lambda it: P, raising=False)
    eng = te.TrainEngine(model, precision)
    monkeypatch.setattr(te, "next", real_next, raising=False)
    final, aux = eng.forward(torch.zeros(shape))
    grads = eng.backward(torch.zeros_like(final), torch.zeros_like(aux))
    trained = {id(p) for n, p in model.named_parameters() if not n.startswith("mobile.classifier")}
    assert set(grads) == trained
    return rec.calls


# the Large case has 128-token attention at 1/32 resolution (256 x 512 input): the tensor-core attention runs too
@pytest.mark.parametrize("mode,C,shape", [("large", 5, (2, 3, 256, 512)), ("small", 8, (2, 3, 64, 96))])
def test_fp16_schedule_mirrors_bf16(monkeypatch, mode, C, shape):
    pos = dtype_positions()
    b16 = record_step(monkeypatch, mode, C, shape, "bf16")
    f16 = record_step(monkeypatch, mode, C, shape, "fp16")
    f16_names = set()
    for name, args in f16:
        assert not (name in TC_NAMES), f"fp16 schedule called the bf16-only {name}"
        dts = [args[i] for i in pos[name]]
        assert all(d in (_lib.F16, _lib.F32) for d in dts), (name, dts)
        if name.endswith("_dt"):
            assert args[-2] == _lib.F16, name   # operand type: the last argument before the stream
        if _lib.F16 in dts:
            f16_names.add(name)
    assert f16_names <= F16_ENTRY_POINTS, f16_names - F16_ENTRY_POINTS
    assert {"cabinet_conv_tc_dt", "cabinet_conv_wgrad_tc_dt", "cabinet_dwconv_tma_dt", "cabinet_im2col_nchw_dt",
            "cabinet_bn_train_stats", "cabinet_bn_train_backward"} <= f16_names
    if mode == "large":
        assert {"cabinet_attn_softmax_dt", "cabinet_conv_tc_imgw_dt", "cabinet_conv_wgrad_tc_batched_dt",
                "cabinet_conv_tc_view_dt"} <= f16_names
    # the same schedule: per entry point as many calls as bf16, once the *_dt names are mapped back
    count16 = Counter(n[:-3] if n.endswith("_dt") else n for n, _ in f16)
    assert count16 == Counter(n for n, _ in b16)
    # and the bf16 schedule itself keeps the old names and never passes fp16
    for name, args in b16:
        assert not name.endswith("_dt") and all(args[i] != _lib.F16 for i in pos[name]), name


def test_train_engine_precision_values():
    from cabinet_b200.engine import dtype_code
    from cabinet_b200.train_engine import TrainEngine

    model = build_model(8, "small")
    with pytest.raises(ValueError):
        TrainEngine(model, "fp8")
    assert dtype_code(torch.float16) == _lib.F16 and dtype_code(torch.bfloat16) == _lib.BF16
    with pytest.raises(TypeError):
        dtype_code(torch.float64)


def _lib_or_skip():
    if not _lib.LIB_PATH.is_file():
        pytest.skip("libcabinet_b200.so is not built")
    return _lib.load()


def test_entry_points_without_fp16_reject_it():
    lib = _lib_or_skip()
    F16 = _lib.F16
    calls = {
        "cabinet_scale_act": lambda: lib.cabinet_scale_act(None, 8, F16, None, 1, 64, 8, 0, 0, None),
        "cabinet_psp_pool": lambda: lib.cabinet_psp_pool(None, 8, F16, None, 1, 8, 8, 8, None, 0, None),
        "cabinet_psp_concat": lambda: lib.cabinet_psp_concat(None, 8, None, None, 40, F16, 1, 8, 8, 8, None),
        "cabinet_softmax_rows": lambda: lib.cabinet_softmax_rows(None, None, F16, 8, 8, None),
        "cabinet_bilinear_nhwc": lambda: lib.cabinet_bilinear_nhwc(None, 8, F16, None, 8, F16, 1, 4, 4, 8, 8, 8, None),
        "cabinet_upsample_logits_nchw": lambda: lib.cabinet_upsample_logits_nchw(None, 1, 4, 4, 8, None, F16, 32, 32, None),
        "cabinet_ohem_ce_forward": lambda: lib.cabinet_ohem_ce_forward(None, F16, None, 0, 1, 8, 64, None, 255, 0.7, 16,
                                                                       None, None, None, None),
        "cabinet_ohem_ce_backward": lambda: lib.cabinet_ohem_ce_backward(None, F16, None, 0, 1, 8, 64, None, None, None,
                                                                         None, None, None),
        "cabinet_dwconv": lambda: lib.cabinet_dwconv(None, 8, None, None, None, 8, F16, 1, 8, 8, 8, 3, 1, 8, 8, 0, None,
                                                     None),
        "cabinet_conv_tc_se (fp16 output)": lambda: lib.cabinet_conv_tc_se(None, 64, 1, 8, 8, 64, None, 0, None, 64, 1, 1, 1,
                                                                           0, None, None, 0, None, F16, 64, 8, 8, 0, None),
        "cabinet_conv_tc_dt (unknown type)": lambda: lib.cabinet_conv_tc_dt(None, 64, 1, 8, 8, 64, None, 64, 1, 1, 1, 0,
                                                                            None, None, 0, None, 0, 64, 8, 8, 0, 7, None),
        "cabinet_add (unknown type)": lambda: lib.cabinet_add(None, 8, None, 8, None, 8, 3, 16, 8, None),
        "cabinet_affine_act (bf16 with fp16)": lambda: lib.cabinet_affine_act(
            ctypes.c_void_p(16), 8, _lib.BF16, None, None, None, 0.0, None, 0, ctypes.c_void_p(16), 8, F16, 16, 16, 8, 0,
            None),
    }
    for what, call in calls.items():
        rc = call()
        msg = lib.cabinet_last_error().decode()
        assert rc == 1 and "element type" in msg, (what, rc, msg)


def test_fp16_tensor_core_kernels_use_tcgen05():
    """The fp16 instantiations of the tensor-core convolution and weight-gradient kernels issue tcgen05.mma (UTCHMMA)."""
    if not _lib.LIB_PATH.is_file():
        pytest.skip("libcabinet_b200.so is not built")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not Path(cuobjdump).is_file():
        pytest.skip("cuobjdump is not installed")
    sass = subprocess.run([cuobjdump, "-sass", str(_lib.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    found = {"conv_tc_kernel": 0, "conv_wgrad_tc_kernel": 0}
    for sec in re.split(r"\n\s*Function : ", sass)[1:]:
        name = sec.split("\n", 1)[0]
        for k in found:
            if re.search(r"\d" + k + r"I.*6__half", name):
                assert "UTCHMMA" in sec, name
                found[k] += 1
    assert found["conv_tc_kernel"] >= 5 and found["conv_wgrad_tc_kernel"] == 1, found

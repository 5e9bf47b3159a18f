"""No GPU: the standalone ContextAggregationBlock's validation, parameter surface and engine housekeeping."""

import copy
import pickle

import pytest
import torch

from cabinet_b200.modules import CABiNet, ContextAggregationBlock

CAB_KEYS = ["gamma"] + [f"global_attn.{m}.{leaf}" for m in ("to_query", "to_key") for leaf in
                        ("0.weight", "1.weight", "1.bias", "1.running_mean", "1.running_var", "1.num_batches_tracked")] + [
    "global_attn.to_value.weight", "global_attn.psp_key.project.weight", "global_attn.psp_value.project.weight",
    "global_attn.project_out.weight"] + [f"local_attn.refine.{i}.block.{leaf}" for i in range(3) for leaf in
                                         ("0.weight", "1.weight", "1.bias", "1.running_mean", "1.running_var",
                                          "1.num_batches_tracked")]


@pytest.mark.parametrize("C,V,what", [(24, 8, "in_channels % 16"), (32, 12, "value_channels % 8"), (40, 16, "% 16")])
def test_widths_outside_the_kernels_raise(C, V, what):
    blk = ContextAggregationBlock(C, V)
    with pytest.raises(ValueError, match=what):
        blk(torch.randn(1, C, 4, 4))


def test_cpu_input_raises():
    with pytest.raises(RuntimeError, match="no CPU path"):
        ContextAggregationBlock(32, 16)(torch.randn(1, 32, 4, 4))


@pytest.mark.parametrize("dtype", [torch.float64, torch.int32])
def test_other_dtypes_raise(dtype):
    with pytest.raises(TypeError, match="float32, bfloat16 or float16"):
        ContextAggregationBlock(32, 16)(torch.zeros(1, 32, 4, 4, dtype=dtype))


def test_wrong_channel_count_raises():
    with pytest.raises(ValueError, match=r"\(N, 32, H, W\)"):
        ContextAggregationBlock(32, 16)(torch.randn(1, 16, 4, 4))


def test_state_dict_keys_unchanged():
    assert list(ContextAggregationBlock(512, 128).state_dict()) == CAB_KEYS
    net_keys = list(CABiNet(5, mode="small").state_dict())
    assert [k[len("ab.a2block."):] for k in net_keys if k.startswith("ab.a2block.")] == CAB_KEYS
    assert all("precision" not in k and "engine" not in k for k in net_keys)


def test_precision_attributes_default_like_cabinet():
    blk, net = ContextAggregationBlock(256, 128), CABiNet(5, mode="small")
    assert (blk.precision, blk.train_precision) == (net.precision, net.train_precision) == ("bf16", "fp32")


def _with_engines(m):
    m.__dict__["_engine"], m.__dict__["_train_engine"] = object(), object()
    return m


def test_deepcopy_and_pickle_carry_no_engine():
    blk = _with_engines(ContextAggregationBlock(64, 32))
    for new in (copy.deepcopy(blk), pickle.loads(pickle.dumps(blk))):
        assert new.__dict__["_engine"] is None and new.__dict__["_train_engine"] is None
        assert new.state_dict().keys() == blk.state_dict().keys()
    assert blk.__dict__["_engine"] is not None   # the original keeps its engines
    net = CABiNet(5, mode="small")
    _with_engines(net.ab.a2block)
    new = copy.deepcopy(net)
    assert new.ab.a2block.__dict__["_engine"] is None and new.ab.a2block.__dict__["_train_engine"] is None


def test_apply_drops_engines():
    blk = _with_engines(ContextAggregationBlock(64, 32))
    blk.float()
    assert blk.__dict__["_engine"] is None and blk.__dict__["_train_engine"] is None
    net = CABiNet(5, mode="small")
    _with_engines(net.ab.a2block)
    net.float()   # the nested block's engines go too
    assert net.ab.a2block.__dict__["_engine"] is None

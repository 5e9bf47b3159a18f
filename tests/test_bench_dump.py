"""CPU: ``bench.py --dump-outputs`` helpers -- float32 arrays, a seeded sample of a large output that is the same from
run to run, at most 64 MB per run."""

import numpy as np
import torch

import bench


def test_small_outputs_are_dumped_whole():
    t = torch.randn(2, 3, 5, dtype=torch.bfloat16)
    a = bench.output_sample(t)
    assert a.dtype == np.float32 and a.shape == (2, 3, 5)
    np.testing.assert_array_equal(a, t.float().numpy())


def test_large_outputs_are_a_fixed_sample(tmp_path):
    n = 64
    t = torch.arange(1000, dtype=torch.float32)
    a, b = bench.output_sample(t, n), bench.output_sample(t.clone(), n)
    assert a.dtype == np.float32 and a.ndim == 1 and n // 2 < len(a) <= n
    np.testing.assert_array_equal(a, b)  # same positions on every run
    assert np.all(np.diff(a) > 0)  # sorted unique flat indices: values of an arange come back in order
    bench.dump_outputs(tmp_path / "d", {"x": a})
    np.testing.assert_array_equal(np.load(tmp_path / "d" / "x.npy"), a)
    # the largest run dumps three sampled outputs and a scalar (--config 5: two logit tensors, gradients, loss)
    assert 4 * bench.DUMP_SAMPLE * 4 <= 64 << 20

"""CPU: the drop-in parameter tree against the reference's, through the weight digests that oracle/make_golden.py
recorded from the imported, unmodified reference (``digest`` of tests/golden/model_*.npz)."""

import numpy as np
import pytest
import torch

from cabinet_b200.synthetic import perturb_state_dict, state_dict_digest

# the reference's digest of its seeded, perturbed weights for each (mode, classes)
REFERENCE_DIGESTS = {("small", 8): "model_small_c8_96x128.npz", ("large", 19): "model_large_c19_64x64.npz"}


@pytest.mark.parametrize("mode,C", [("small", 8), ("large", 19)])
def test_state_dict_bit_identical(golden_dir, mode, C):
    """``torch.manual_seed(0)`` then construction: the same keys in the same order and the same bytes as the reference.

    The digest covers keys and raw bytes after ``perturb_state_dict``, which overwrites BN statistics / affine, biases
    and ``gamma``.  Every other tensor is compared as initialised.  Construction draws all parameters from one seeded
    stream, so a bias that differs in presence, shape or order also shifts every later weight."""
    from cabinet_b200 import BACKBONE_CFGS, CABiNet

    g = np.load(golden_dir / REFERENCE_DIGESTS[(mode, C)])
    assert (str(g["mode"]), int(g["n_classes"])) == (mode, C)
    torch.manual_seed(0)
    sd = CABiNet(C, mode=mode, cfgs=BACKBONE_CFGS[mode]).state_dict()
    assert state_dict_digest(perturb_state_dict(sd)) == str(g["digest"])

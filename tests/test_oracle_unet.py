"""Pins oracle/unet_ref.py against golden vectors produced by the reference modules
(tests/golden/make_unet_golden.py): the reduced config, and the full-width projector at grid 16, where the
generator also checked the oracle bit-for-bit against the reference before storing the reference's output."""
import os

import numpy as np
import pytest
import torch

from oracle import unet_ref as O

GOLD = os.path.join(os.path.dirname(__file__), "golden", "unet_small.npz")
GOLD_G16 = os.path.join(os.path.dirname(__file__), "golden", "unet_ref_g16.npz")


def _small(out, seed):
    net = (O.RegressionUNet if out == 3 else O.SegmentationUNet)(64, 32, 64, 3, (1, 1, 2, 4), (), 8, out).eval()
    net.load_state_dict(O.seeded_state_dict(net, seed))
    return net


@pytest.mark.parametrize("name,out", [("reg", 3), ("seg", 8)])
def test_oracle_matches_golden(name, out):
    g = np.load(GOLD)
    net = _small(out, int(g[f"{name}_seed"]))
    torch.set_num_threads(1)
    with torch.no_grad():
        y = net(torch.from_numpy(g["x"]))
    # same torch ops in the same order: agreement to fp32 round-off across torch builds / ISAs
    assert np.abs(y.numpy() - g[f"{name}_y"]).max() < 2e-5
    assert np.abs(g[f"{name}_y"]).max() > 0.5        # non-vacuous: zero_module'd tensors were re-seeded


def test_fresh_reference_like_network_is_zero():
    """SURVEY fact 3: default initialisation gives exactly 0, hence the seeded parameters."""
    net = O.RegressionUNet(64, 32, 64, 3, (1, 1, 2, 4), (), 8, 3).eval()
    with torch.no_grad():
        y = net(O.synthetic_features(1, 64, 8, seed=0))
    assert float(y.abs().max()) == 0.0


def test_oracle_matches_reference_modules():
    g = np.load(GOLD_G16)
    mine = O.RegressionUNet(96, 32, 64, 3, (1, 1, 2, 4), (), 16, 3).eval()
    assert list(mine.state_dict().keys()) == list(g["keys"])
    mine.load_state_dict(O.seeded_state_dict(mine, int(g["seed"])))
    x = O.synthetic_features(1, 96, 16, seed=int(g["x_seed"]))
    torch.set_num_threads(1)
    with torch.no_grad():
        y = mine(x)
    # bit-identical where the vectors were made; another CPU or thread count reorders the fp32 sums
    assert np.abs(y.numpy() - g["y"]).max() < 2e-5
    assert np.abs(g["y"]).max() > 0.5


def test_light_projector_and_no_projector_variants():
    """feature types rgb/occupancy use the single-layer projector; feature_channels == cond_dim uses none
    (training_discrete.py:62-68)."""
    for C in (3, 32):
        net = O.SegmentationUNet(C, 32, 64, 1, (1, 2), (), 8, 8).eval()
        net.load_state_dict(O.seeded_state_dict(net, 1))
        with torch.no_grad():
            y = net(O.synthetic_features(1, C, 8, seed=2, scale=1.0))
        assert y.shape == (1, 8, 8, 8, 8) and torch.isfinite(y).all()
        assert (net.projector is None) == (C == 32)

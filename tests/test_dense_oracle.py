"""CPU: pins oracle/torch_dense.py (the plain-PyTorch restatement used as the dense oracle on the GPU box) to
(a) the golden outputs produced from the unmodified reference modules, using the drop-in modules purely as parameter
containers, and (b) the parameter names and shapes of the reference modules."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import torch_dense as TD
from oracle.make_golden_dense import GATES_ALL, GATES_PERCEIVE, STATE_DICTS, dense_input, state_dict_shapes
from stp3_b200.models.decoder import Decoder
from stp3_b200.models.temporal_model import TemporalModel
from tests.helpers import GOLDEN


def load(name):
    return dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))


def temporal_input(g):
    x = dense_input((1, 3, 70, int(g["H"]), int(g["W"])), int(g["in_seed"]))
    x[:, :, 64:] = x[:, :, 64:, :1, :1]
    return x


def test_temporal_model_restatement_matches_reference_output():
    g = load("dense_temporal_model.npz")
    with torch.no_grad():
        tm = TD.init_exact(TemporalModel(70, 3, (int(g["H"]), int(g["W"])), start_out_channels=64), seed=int(g["seed"])).eval()
        y = TD.temporal_model(temporal_input(g), tm)
    ref = torch.from_numpy(g["out"])
    assert (y - ref).abs().max() <= 2e-5 * ref.abs().max()


def test_temporal_model_restatement_matches_reference_output_stress_shape():
    """BASELINE configs[4] shape: 134 input channels (128 + ego-motion), receptive field 5 (four blocks)."""
    g = load("dense_temporal_model_stress.npz")
    H, W = int(g["H"]), int(g["W"])
    with torch.no_grad():
        tm = TD.init_exact(TemporalModel(134, 5, (H, W), start_out_channels=64), seed=int(g["seed"])).eval()
        x = dense_input((1, 5, 134, H, W), int(g["in_seed"]))
        x[:, :, 128:] = x[:, :, 128:, :1, :1]
        y = TD.temporal_model(x, tm)
    ref = torch.from_numpy(g["out"])
    assert y.shape == ref.shape and (y - ref).abs().max() <= 2e-5 * ref.abs().max()


@pytest.mark.parametrize("name,gates", [("perceive", GATES_PERCEIVE), ("all", GATES_ALL)])
def test_decoder_restatement_matches_reference_output(name, gates):
    g = load(f"dense_decoder_{name}.npz")
    with torch.no_grad():
        dec = TD.init_exact(Decoder(64, 2, 3, 2, gates), seed=int(g["seed"])).eval()
        out = TD.decoder(dense_input((1, 3, 64, int(g["H"]), int(g["W"])), int(g["in_seed"])), dec)
    for k, v in out.items():
        if v is None:
            assert k not in g
            continue
        ref = torch.from_numpy(g[k])
        assert v.shape == ref.shape, k
        assert (v - ref).abs().max() <= 5e-5 * max(1.0, float(ref.abs().max())), k   # fp32 op-order noise


def test_state_dict_keys_match_reference_when_available():
    """The drop-in modules keep the reference's checkpoint layout: the same parameter and buffer names with the same
    shapes as the reference modules had (tests/golden/reference_state_dicts.json, oracle/make_golden_dense.py), so a
    reference checkpoint loads into them strictly and theirs into the reference."""
    with open(os.path.join(GOLDEN, STATE_DICTS)) as f:
        ref = json.load(f)
    assert state_dict_shapes(TemporalModel(70, 3, (20, 20))) == ref["temporal_model"]
    assert state_dict_shapes(Decoder(64, 2, 3, 2, GATES_ALL)) == ref["decoder_all"]

"""Generates tests/golden/dense_*.npz from the UNMODIFIED reference modules (TemporalModel, Decoder) run on CPU in the
build container with deterministic weights (oracle.torch_dense.init_exact) and inputs, and
tests/golden/reference_state_dicts.json (the parameter names and shapes of those modules).  Test infrastructure; run
by hand:  python -m oracle.make_golden_dense"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.ref_loader import load_reference  # noqa: E402
from oracle import torch_dense as TD  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
GATES_PERCEIVE = dict(perceive_hdmap=True, predict_pedestrian=True, predict_instance=False, predict_future_flow=False,
                      planning=False)
GATES_ALL = dict(perceive_hdmap=True, predict_pedestrian=True, predict_instance=True, predict_future_flow=True,
                 planning=True)


def dense_input(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return TD.exact_gauss(shape, g)


STATE_DICTS = "reference_state_dicts.json"


def state_dict_shapes(module):
    return {k: list(v.shape) for k, v in module.state_dict().items()}


def write_state_dicts(ref):
    """The checkpoint layout the drop-in modules must keep: TemporalModel(70, 3, (20, 20)) and the decoder with every
    head on, Decoder(64, 2, 3, 2, GATES_ALL)."""
    rec = {"temporal_model": state_dict_shapes(ref.temporal_model.TemporalModel(70, 3, (20, 20))),
           "decoder_all": state_dict_shapes(ref.decoder.Decoder(64, 2, 3, 2, GATES_ALL))}
    with open(os.path.join(OUT, STATE_DICTS), "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")


def main():
    ref = load_reference()
    write_state_dicts(ref)
    torch.manual_seed(0)
    H, W = 24, 40
    with torch.no_grad():
        tm = TD.init_exact(ref.temporal_model.TemporalModel(70, 3, (H, W), start_out_channels=64), seed=1).eval()
        x = dense_input((1, 3, 70, H, W), 5)
        x[:, :, 64:] = x[:, :, 64:, :1, :1]          # the six ego-motion channels are spatially constant (stp3.py:148)
        y = tm(x)
        np.savez_compressed(os.path.join(OUT, "dense_temporal_model.npz"), out=y.numpy(), H=H, W=W, seed=1, in_seed=5)
        print("temporal_model", tuple(y.shape), float(y.abs().max()))
        # stress shape (BASELINE configs[4]): 128 + 6 input channels, receptive field 5 -> four blocks, the first with
        # 67-channel paths
        Hs, Ws = 16, 24
        tms = TD.init_exact(ref.temporal_model.TemporalModel(134, 5, (Hs, Ws), start_out_channels=64), seed=3).eval()
        xs = dense_input((1, 5, 134, Hs, Ws), 7)
        xs[:, :, 128:] = xs[:, :, 128:, :1, :1]
        ys = tms(xs)
        np.savez_compressed(os.path.join(OUT, "dense_temporal_model_stress.npz"), out=ys.numpy(), H=Hs, W=Ws, seed=3,
                            in_seed=7)
        print("temporal_model (stress shape)", tuple(ys.shape), float(ys.abs().max()))
        for name, gates in (("perceive", GATES_PERCEIVE), ("all", GATES_ALL)):
            dec = TD.init_exact(ref.decoder.Decoder(64, 2, 3, 2, gates), seed=2).eval()
            x = dense_input((1, 3, 64, H, W), 6)
            out = dec(x)
            rec = {k: v.numpy() for k, v in out.items() if v is not None}
            np.savez_compressed(os.path.join(OUT, f"dense_decoder_{name}.npz"), H=H, W=W, seed=2, in_seed=6, **rec)
            print("decoder", name, {k: tuple(v.shape) for k, v in rec.items()})


if __name__ == "__main__":
    main()

"""Fixture for the network layout tests: the state-dict layout of the reference's Seg_Model (networks/ccnet.py:199-205,
num_classes=19, recurrence=2) built from the reference's own networks/ccnet.py and cc_attention package, with the harness's
inplace_abn stand-in for the native extension the reference does not vendor.  Only key names and shapes are stored.

    python tests/golden/make_network_golden.py <reference tree>      (writes tests/golden/ccnet_state_dict.npz)
"""
import importlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def main(ref):
    if not os.path.exists(os.path.join(ref, "networks", "ccnet.py")):
        sys.exit(f"{ref}: not a reference tree (networks/ccnet.py missing)")
    # the reference tree first (its own cc_attention, networks, utils), then the inplace_abn stand-in
    sys.path[:0] = [ref, os.path.join(ROOT, "harness", "shims")]
    ccnet = importlib.import_module("networks.ccnet")
    assert ccnet.__file__.startswith(os.path.abspath(ref)) and ccnet.CrissCrossAttention.__module__.startswith("cc_attention")
    with torch.device("meta"):
        model = ccnet.Seg_Model(num_classes=19, recurrence=2)
    sd = model.state_dict()
    shapes = np.full((len(sd), 4), -1, dtype=np.int64)          # -1 pads the unused trailing dimensions
    for i, v in enumerate(sd.values()):
        shapes[i, :v.dim()] = v.shape
    out = {"keys": np.array(list(sd)), "shapes": shapes, "ndim": np.array([v.dim() for v in sd.values()]),
           "n_params": np.int64(sum(p.numel() for p in model.parameters())), "recurrence": np.int64(model.recurrence)}
    np.savez_compressed(os.path.join(HERE, "ccnet_state_dict.npz"), **out)
    print(len(sd), "tensors,", int(out["n_params"]), "parameters")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])

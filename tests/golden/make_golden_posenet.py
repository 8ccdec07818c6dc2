#!/usr/bin/env python
"""State dict of the reference's PoseNet (lib/models/posenet.py:41-98) as the UNMODIFIED reference constructs it:

    python tests/golden/make_golden_posenet.py      ->  tests/golden/posenet_state_dict.npz

  keys           the state_dict keys in the reference's order
  sd/<key>       every tensor of posenet.get_model(17, hid_dim=64, num_layer=2, p_dropout=0.5) under torch.manual_seed(5)
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_shim  # noqa: E402


def main():
    ref_shim.load("human36")
    from models import posenet  # noqa: E402  (reference module)

    torch.manual_seed(5)
    net = posenet.get_model(17, hid_dim=64, num_layer=2, p_dropout=0.5, pretrained=False)
    sd = net.state_dict()
    out = {"keys": np.array(list(sd.keys()))}
    for k, v in sd.items():
        out["sd/" + k] = v.numpy()
    path = os.path.join(HERE, "posenet_state_dict.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()

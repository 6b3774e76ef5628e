"""Shared test helpers (config objects, comparison utilities)."""
import json
import os
import types

import numpy as np

from yolact_b200.config import CONFIGS


def cfg_for(name):
    return CONFIGS[name].copy()


def unpack_masks(packed, w):
    return np.unpackbits(packed, axis=-1)[..., :w].astype(np.float32)


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-12))


def load_reference_cfgs():
    """The reference's published configs as duck-typed cfg objects (attribute access, backbone.type a class of the
    stored name), rebuilt from tests/golden/reference_cfgs.json: the fields yolact_b200.config.from_reference_cfg
    reads, written by oracle/gen_golden.py from the reference tree."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_cfgs.json")) as f:
        raw = json.load(f)
    out = {}
    for name, d in raw.items():
        b = dict(d["backbone"], type=type(d["backbone"]["type"], (), {}),
                 transform=types.SimpleNamespace(**d["backbone"]["transform"]))
        out[name] = types.SimpleNamespace(**dict(d, backbone=types.SimpleNamespace(**b),
                                                 fpn=types.SimpleNamespace(**d["fpn"])))
    return out

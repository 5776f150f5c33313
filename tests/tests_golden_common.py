import os

import numpy as np

from conftest import DATA_DIR, GOLDEN_DIR

RENDERS = {"c1_whitted": "c1_torusknot", "c2_reflective": "c2_monkey", "c2_null": "c2_monkey_null",
           "mix_deterministic": "deterministic_mix", "c3_preview": "c3_unitychan", "c3_path": "c3_unitychan",
           "default_path": "default_scene"}


def golden(name):
    """A committed fixture.  Those of scenes with meshes come from the reference's own meshes where they are
    staged, else from the generated stand-ins (tests/golden/standin/, make_golden.py --standin)."""
    d = GOLDEN_DIR if name == "kat" or os.path.isdir(DATA_DIR) else os.path.join(GOLDEN_DIR, "standin")
    path = os.path.join(d, name + ".npz")
    assert os.path.exists(path), f"{path} missing (tests/golden/make_golden.py)"
    return np.load(path)

#!/usr/bin/env python
"""Write tests/golden/model_tables.npz: the model tables a fresh parse of the reference's MJCF files yields (the in-repo parser,
smplsim_b200/mjcf.py, on the XMLs tools/extract_model.py derives the shipped assets from).  Needs a checkout of the reference:

    python tests/golden/make_golden_model_tables.py <reference checkout>

Keys are "<model>.<field>"; the name lists are stored as unicode arrays so that np.load needs no pickle.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
from smplsim_b200.model import load_model  # noqa: E402

XMLS = {"smpl": "smpl_sim/data/assets/mjcf/smpl_humanoid.xml", "smplx": "smpl_humanoid.xml"}
NAMES = ("body_names", "joint_names", "geom_names")
FIELDS = ("body_parent", "body_pos", "body_quat", "body_mass", "body_ipos", "body_inertia", "dof_armature", "dof_range", "dof_invweight0",
          "geom_type", "geom_body", "geom_pos", "geom_mat", "geom_size", "act_kp", "act_kd", "act_torque_lim", "act_scale", "act_offset")

if __name__ == "__main__":
    ref = sys.argv[1]
    out = {}
    for name, rel in XMLS.items():
        m = load_model(os.path.join(ref, rel))
        for f in NAMES:
            out[f"{name}.{f}"] = np.array(getattr(m, f), dtype=str)
        for f in FIELDS:
            out[f"{name}.{f}"] = np.asarray(getattr(m, f))
    np.savez_compressed(os.path.join(HERE, "model_tables.npz"), **out)
    print("model_tables.npz:", {name: int(out[f"{name}.body_mass"].shape[0]) for name in XMLS})

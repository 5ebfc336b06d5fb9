"""The shipped constant tables (smplsim_b200/assets/*.model.json) are *derived* from the reference's MJCF files by the in-repo parser
(tools/extract_model.py).  They must equal what a fresh parse of those XMLs gave (tests/golden/model_tables.npz, written by
tests/golden/make_golden_model_tables.py); the MJCF parser itself is exercised on a small hand-written model."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from smplsim_b200.mjcf import parse_mjcf
from smplsim_b200.model import build_model, load_model

FIELDS = ("body_parent", "body_pos", "body_quat", "body_mass", "body_ipos", "body_inertia", "dof_armature", "dof_range", "dof_invweight0",
          "geom_type", "geom_body", "geom_pos", "geom_mat", "geom_size", "act_kp", "act_kd", "act_torque_lim", "act_scale", "act_offset")


@pytest.mark.parametrize("name", ["smpl", "smplx"])
def test_shipped_tables_equal_fresh_parse_of_reference_xml(name):
    g = np.load(os.path.join(GOLDEN, "model_tables.npz"))
    a = load_model(name)
    for f in ("body_names", "joint_names", "geom_names"):
        assert list(getattr(a, f)) == g[f"{name}.{f}"].tolist(), f
    for f in FIELDS:
        x, y = np.asarray(getattr(a, f)), g[f"{name}.{f}"]
        assert x.shape == y.shape and np.allclose(x, y, rtol=0, atol=1e-12), f


MINI = """
<mujoco model="mini">
  <compiler coordinate="local"/>
  <default><joint damping="0" armature="0.01" stiffness="0" limited="true"/><geom condim="3" margin="0.001"/></default>
  <worldbody>
    <geom name="floor" type="plane" pos="0 0 0" size="100 100 0.2"/>
    <body name="Pelvis" pos="0 0 1">
      <freejoint name="Pelvis"/>
      <geom name="Pelvis" type="sphere" size="0.1" density="1000"/>
      <body name="L_Hip" pos="0 0.1 -0.1">
        <joint name="L_Hip_x" type="hinge" axis="1 0 0" range="-90 90"/>
        <joint name="L_Hip_y" type="hinge" axis="0 1 0" range="-180 180"/>
        <joint name="L_Hip_z" type="hinge" axis="0 0 1" range="-45 45"/>
        <geom name="L_Hip" type="capsule" fromto="0 0 0 0 0 -0.4" size="0.05" density="1000"/>
        <body name="L_Knee" pos="0 0 -0.4">
          <joint name="L_Knee_x" type="hinge" axis="1 0 0" range="-180 180"/>
          <joint name="L_Knee_y" type="hinge" axis="0 1 0" range="-180 180"/>
          <joint name="L_Knee_z" type="hinge" axis="0 0 1" range="-180 180"/>
          <geom name="L_Knee" type="box" pos="0 0 -0.1" size="0.05 0.04 0.1" density="500"/>
        </body>
      </body>
    </body>
  </worldbody>
  <actuator>
    <motor name="L_Hip_x" joint="L_Hip_x" gear="1"/><motor name="L_Hip_y" joint="L_Hip_y" gear="1"/><motor name="L_Hip_z" joint="L_Hip_z" gear="1"/>
    <motor name="L_Knee_x" joint="L_Knee_x" gear="1"/><motor name="L_Knee_y" joint="L_Knee_y" gear="1"/><motor name="L_Knee_z" joint="L_Knee_z" gear="1"/>
  </actuator>
</mujoco>
"""


def test_mjcf_parser_masses_inertias_ranges_on_a_hand_model():
    """Geom -> inertia rules of SURVEY A.1: sphere, capsule from fromto, box; degrees -> radians; tree order."""
    p = parse_mjcf(MINI)
    m = build_model(p, contact_bodies=["L_Knee"])
    assert m.body_names == ["Pelvis", "L_Hip", "L_Knee"] and list(m.body_parent) == [-1, 0, 1]
    assert (m.nq, m.nv, m.nu) == (13, 12, 6)
    r, H, rho = 0.05, 0.4, 1000.0
    m_sph = rho * 4 / 3 * np.pi * 0.1 ** 3
    m_cyl, m_cap = rho * np.pi * r * r * H, rho * 4 / 3 * np.pi * r ** 3
    m_box = 500.0 * 8 * 0.05 * 0.04 * 0.1
    assert np.allclose(m.body_mass, [m_sph, m_cyl + m_cap, m_box], rtol=1e-12)
    assert np.allclose(m.body_ipos[1], [0, 0, -0.2]) and np.allclose(m.body_ipos[2], [0, 0, -0.1])
    Izz = m_cyl * r * r / 2 + 0.4 * m_cap * r * r
    Ixx = m_cyl * (3 * r * r + H * H) / 12 + m_cap * (0.4 * r * r + 0.375 * r * H + 0.25 * H * H)
    I1 = np.sort(np.asarray(m.body_inertia[1])[:3])
    assert np.allclose(I1, np.sort([Ixx, Ixx, Izz]), rtol=1e-9)
    bx = m_box / 3 * np.array([0.04 ** 2 + 0.1 ** 2, 0.05 ** 2 + 0.1 ** 2, 0.05 ** 2 + 0.04 ** 2])
    assert np.allclose(np.sort(np.asarray(m.body_inertia[2])[:3]), np.sort(bx), rtol=1e-9)
    assert np.allclose(m.dof_range[6], [-np.pi / 2, np.pi / 2]) and np.allclose(m.dof_range[8], [-np.pi / 4, np.pi / 4])
    assert np.allclose(m.dof_armature, [0] * 6 + [0.01] * 6)

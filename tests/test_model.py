"""Model table known answers (SURVEY Appendix A) and the URDF parser."""
import json
import os

import numpy as np
import pytest

from solorl_b200.abi import model_table
from solorl_b200.model import JOINT_FIXED, JOINT_REVOLUTE, SoloModel
from tests.helpers import GOLDEN


def test_solo8_table():
    m = SoloModel.builtin("solo8")
    assert m.num_links == 12 and m.nj == 8
    assert m.joints_idx == [0, 1, 3, 4, 6, 7, 9, 10]          # solo.py:99-106 on solo.urdf
    assert m.feet_idx == [2, 5, 8, 11]
    assert m.ordered_joint_names == ["FL_HFE", "FL_KFE", "FR_HFE", "FR_KFE", "HL_HFE", "HL_KFE", "HR_HFE", "HR_KFE"]
    assert abs(m.total_mass - 2.17784899) < 1e-8
    assert m.base_mass == pytest.approx(1.43315091)
    assert np.allclose(m.base_inertia, [0.00578574, 0, 0, 0.01938108, 0, 0.02476124])
    assert m.joint_state_limit == 10.0                        # solo.urdf:47, solo.py:109
    assert np.allclose(m.origin[0], [0.19, 0.1046, 0]) and np.allclose(m.axis[0], [0, 1, 0])
    assert np.allclose(m.origin[1], [0, 0.03745, -0.16])
    assert np.allclose(m.origin[2], [0, 0.008, -0.16]) and m.jtype[2] == JOINT_FIXED


def test_solo12_table():
    m = SoloModel.builtin("solo12")
    assert m.num_links == 16 and m.nj == 12
    assert m.joints_idx == [0, 1, 2, 4, 5, 6, 8, 9, 10, 12, 13, 14]
    assert m.feet_idx == [3, 7, 11, 15]
    assert m.ordered_joint_names[:3] == ["FL_HAA", "FL_HFE", "FL_KFE"]
    assert abs(m.total_mass - 2.50000279) < 1e-8
    assert np.allclose(m.axis[0], [1, 0, 0]) and np.allclose(m.axis[1], [0, 1, 0])
    assert np.allclose(m.origin[0], [0.1946, 0.0875, 0])
    assert all(t == JOINT_REVOLUTE for i, t in enumerate(m.jtype) if i not in m.feet_idx)
    # lower-leg COM y is +0.00787644 on BOTH sides (a quirk of the URDF, SURVEY Appendix A)
    assert m.com[2][1] == pytest.approx(0.00787644) and m.com[6][1] == pytest.approx(0.00787644)


def test_model_table_struct_roundtrip():
    m = SoloModel.builtin("solo12")
    t = model_table(m)
    assert t.num_links == 16 and t.num_feet == 4
    assert list(t.foot_link)[:4] == [3, 7, 11, 15]
    assert t.parent[0] == -1 and t.parent[1] == 0 and t.parent[3] == 2
    assert t.foot_radius == pytest.approx(0.016)


def test_urdf_parser_on_synthetic(tmp_path):
    urdf = """<?xml version="1.0"?><robot name="r">
      <link name="base"><inertial><origin xyz="0 0 0" rpy="0 0 0"/><mass value="2"/>
        <inertia ixx="1" ixy="0" ixz="0" iyy="2" iyz="0" izz="3"/></inertial></link>
      <joint name="A_HFE" type="revolute"><parent link="base"/><child link="a"/>
        <axis xyz="0 1 0"/><origin xyz="0.1 0.2 0" rpy="0 0 0"/><limit lower="-7" upper="7" effort="1" velocity="1"/></joint>
      <link name="a"><inertial><origin xyz="0 0 -0.1" rpy="0 0 0"/><mass value="0.5"/>
        <inertia ixx="0.1" ixy="0.01" ixz="0" iyy="0.2" iyz="0.02" izz="0.3"/></inertial></link>
      <joint name="A_ANKLE" type="fixed"><parent link="a"/><child link="f"/><origin xyz="0 0 -0.2" rpy="0 0 0"/></joint>
      <link name="f"><inertial><mass value="0.1"/><inertia ixx="1e-3" ixy="0" ixz="0" iyy="1e-3" iyz="0" izz="1e-3"/></inertial></link>
    </robot>"""
    p = tmp_path / "r.urdf"
    p.write_text(urdf)
    m = SoloModel.from_urdf(str(p))
    assert m.joint_names == ["A_HFE", "A_ANKLE"] and m.joints_idx == [0] and m.feet_idx == [1]
    assert m.parent == [-1, 0] and m.total_mass == pytest.approx(2.6)
    assert np.allclose(m.inertia[0], [0.1, 0.01, 0, 0.2, 0.02, 0.3])
    assert m.joint_state_limit == 7.0


def test_urdf_parser_rejects_rpy(tmp_path):
    p = tmp_path / "bad.urdf"
    p.write_text("""<robot name="r"><link name="b"/><link name="c"/>
      <joint name="j" type="revolute"><parent link="b"/><child link="c"/><origin xyz="0 0 0" rpy="0 0.1 0"/></joint></robot>""")
    with pytest.raises(ValueError):
        SoloModel.from_urdf(str(p))


def test_resolve_reference_config_paths():
    # configs/basic.yaml:4 carries the reference author's absolute path
    m = SoloModel.resolve("/home/maractin/Workspace/soloRL/solo_description/robots/solo.urdf")
    assert m.nj == 8
    m = SoloModel.resolve("/home/maractin/Workspace/soloRL/solo_description/robots/solo12.urdf")
    assert m.nj == 12
    with pytest.raises(FileNotFoundError):
        SoloModel.resolve("/nowhere/other.urdf")


@pytest.mark.parametrize("urdf,name", [("solo.urdf", "solo8"), ("solo12.urdf", "solo12")])
def test_builtin_equals_reference_urdf(urdf, name):
    # the fields SoloModel.from_urdf reads off the reference's solo_description/robots/<urdf>, stored as golden data
    with open(os.path.join(GOLDEN, "reference_urdf_models.json")) as f:
        a = json.load(f)[urdf]
    b = SoloModel.builtin(name)
    assert a["joint_names"] == b.joint_names and a["parent"] == b.parent and a["jtype"] == b.jtype
    for f in ("axis", "origin", "mass", "com", "inertia", "base_inertia"):
        assert np.array_equal(np.array(a[f], dtype=np.float64), getattr(b, f)), f

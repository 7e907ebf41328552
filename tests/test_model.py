"""MJCF reader: the committed mesh-free scene carries the reference's numbers (SURVEY.md Appendix A)."""
import os

import numpy as np
import pytest

from conftest import ROOT
from so100_mujoco_rl_b200.model import euler_to_quat, load_model, quat_to_mat


def test_chain_constants(spec):
    assert spec.joint_names == ["Rotation", "Pitch", "Elbow", "Wrist_Pitch", "Wrist_Roll", "Jaw"]
    assert np.isclose(spec.body_mass.sum(), 0.6089654, atol=1e-7)
    assert np.allclose(spec.jnt_range, [[-2.2, 2.2], [-3.14158, 0.2], [0, 3.14158], [-2.0, 1.8], [-3.14158, 3.14158], [-0.2, 2.0]])
    assert np.allclose(spec.jnt_axis, [[0, 1, 0], [1, 0, 0], [1, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]])
    assert (spec.jnt_armature == 0.1).all() and (spec.jnt_frictionloss == 0.1).all()
    assert (spec.act_kp == 50).all() and (spec.act_dampratio == 1).all()
    assert np.allclose(spec.act_forcerange, [[-35, 35]] * 6) and np.allclose(spec.act_ctrlrange, [[-3.14158, 3.14158]] * 6)
    assert spec.nsubstep == 16 and spec.timestep == 0.002 and spec.cam_fovy_deg == 120
    assert spec.cam_body == 4 and np.allclose(spec.cam_pos, [-0.001, -0.023827, 0.05778])
    assert np.allclose(spec.jnt_solref_limit, [[0.02, 1]] * 6) and np.allclose(spec.dof_solimp_friction[:, :3], [[0.9, 0.95, 0.001]] * 6)


def test_euler_is_intrinsic_xyz():
    q = euler_to_quat([0.3, -0.7, 1.1])
    cx, sx, cy, sy, cz, sz = np.cos(0.3), np.sin(0.3), np.cos(-0.7), np.sin(-0.7), np.cos(1.1), np.sin(1.1)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    assert np.allclose(quat_to_mat(q), Rx @ Ry @ Rz, atol=1e-14)


def test_asset_equals_reference_mjcf(spec):
    """tests/golden/ref_mjcf.npz: the reference's env01.xml as load_model reads it (tools/gen_golden_from_reference.py)."""
    ref = np.load(os.path.join(ROOT, "tests", "golden", "ref_mjcf.npz"))
    for f in ("body_pos", "body_quat", "body_ipos", "body_iquat", "body_mass", "body_inertia", "jnt_axis", "jnt_range",
              "jnt_armature", "jnt_frictionloss", "act_kp", "act_dampratio", "act_ctrlrange", "act_forcerange",
              "cam_pos", "cam_quat", "ee_offset", "gravity"):
        assert np.array_equal(getattr(spec, f), ref[f]), f
    assert spec.cam_fovy_deg == ref["cam_fovy_deg"] and spec.timestep == ref["timestep"]


def test_unsupported_models_are_rejected(tmp_path, spec):
    import so100_mujoco_rl_b200.model as M
    txt = open(M.ASSET_SCENE).read().replace('<joint name="so100_Jaw" class="Jaw"/>', '<joint name="so100_Jaw" class="Jaw" type="slide"/>')
    p = tmp_path / "bad.xml"
    p.write_text(txt)
    with pytest.raises(ValueError):
        load_model(str(p))

"""Model compiler (URDF / TOML -> flat tables): Pinocchio joint ordering and indexing, fixed-joint
merging, hardware description semantics (robot.py:518-847), compiled BASELINE robots."""
import json
import os

import numpy as np
import pytest

from jiminy_b200 import model as M
from jiminy_b200 import robots as R

from conftest import DATA, ROOT

# the reference's ANYmal description (ANYbotics' anymal.urdf and jiminy's anymal_hardware.toml), kept as test inputs
REF_ANYMAL = os.path.join(ROOT, "tests", "golden", "anymal")


def test_simple_pendulum_fixed_joint_merge():
    r = M.build_robot_table(os.path.join(DATA, "simple_pendulum.urdf"), has_freeflyer=False)
    assert r.joint_names == ["universe", "PendulumJoint"]
    assert r.nq == 1 and r.nv == 1 and int(r.joint_type[1]) == M.JB_JOINT_RY
    # the 5 kg mass hangs 1 m along z after the fixed joint: merged into the joint's body
    np.testing.assert_allclose(r.inertia[1, :4], [5.0, 0.0, 0.0, 1.0])
    assert r.frames["PendulumLink"].joint == 1
    np.testing.assert_allclose(r.frames["PendulumLink"].placement.p, [0, 0, 1.0])


def test_branched_arm_ordering_and_types():
    r = M.build_robot_table(os.path.join(DATA, "branched_arm.urdf"), has_freeflyer=True)
    # children visited in alphabetical joint-name order, depth first
    assert r.joint_names == ["universe", "root_joint", "a_shoulder", "a_elbow", "a_spin", "b_hip", "b_slide",
                             "b_skew_slide", "b_ankle_z", "c_spin_skew"]
    t = dict(zip(r.joint_names, r.joint_type.tolist()))
    assert t["root_joint"] == M.JB_JOINT_FREEFLYER and t["a_shoulder"] == M.JB_JOINT_RX
    assert t["a_elbow"] == M.JB_JOINT_RY and t["a_spin"] == M.JB_JOINT_RUBZ and t["b_hip"] == M.JB_JOINT_RU
    assert t["b_slide"] == M.JB_JOINT_PZ and t["b_skew_slide"] == M.JB_JOINT_PU
    assert t["b_ankle_z"] == M.JB_JOINT_RZ and t["c_spin_skew"] == M.JB_JOINT_RUBU
    assert r.nq == 7 + 2 + 2 + 4 + 2 and r.nv == 6 + 2 + 1 + 4 + 1
    assert list(r.idx_q) == [0, 0, 7, 8, 9, 11, 12, 13, 14, 15] and list(r.idx_v) == [0, 0, 6, 7, 8, 9, 10, 11, 12, 13]
    np.testing.assert_allclose(np.linalg.norm(r.axis[5]), 1.0)
    # total mass is conserved by the fixed-joint merge
    np.testing.assert_allclose(r.mass, 4.0 + 1.2 + 0.8 + 0.3 + 0.2 + 1.5 + 0.9 + 0.4 + 0.1 + 0.5)
    file_order = M.build_robot_table(os.path.join(DATA, "branched_arm.urdf"), True, joint_order="file")
    assert file_order.joint_names[2] == "a_shoulder" and file_order.joint_names[-1] == "c_spin_skew"


def test_inertia_merge_parallel_axis():
    a = M.Inertia(2.0, np.array([0.1, 0.0, 0.0]), np.diag([0.01, 0.02, 0.03]))
    b = M.Inertia(3.0, np.array([-0.2, 0.1, 0.0]), np.diag([0.02, 0.01, 0.04]))
    s = a + b

    def about_origin(y):
        c = y.lever
        return y.I + y.mass * (np.dot(c, c) * np.eye(3) - np.outer(c, c))
    np.testing.assert_allclose(about_origin(s), about_origin(a) + about_origin(b), atol=1e-15)
    np.testing.assert_allclose(s.lever, (2.0 * a.lever + 3.0 * b.lever) / 5.0)


@pytest.mark.parametrize("name", R.ROBOT_NAMES)
def test_compiled_robots_load(name):
    robot, opt = R.load_robot(name)
    M.validate_options(R.baseline_options(name, opt))
    d = M.robot_table_to_dict(robot)
    again = M.robot_table_from_dict(json.loads(json.dumps(d)))
    np.testing.assert_array_equal(again.placement, robot.placement)
    assert again.joint_names == robot.joint_names and len(again.motors) == robot.nmotors


def test_anymal_facts():
    """SURVEY.md App. C: joint order, motor order = TOML order, contact frames sorted by name."""
    r, opt = R.load_robot("anymal")
    assert r.joint_names == ["universe", "root_joint", "LF_HAA", "LF_HFE", "LF_KFE", "LH_HAA", "LH_HFE", "LH_KFE",
                             "RF_HAA", "RF_HFE", "RF_KFE", "RH_HAA", "RH_HFE", "RH_KFE"]
    assert (r.nq, r.nv, r.nmotors) == (19, 18, 12)
    assert [m.name for m in r.motors][:6] == ["LF_HAA", "LF_HFE", "LF_KFE", "RF_HAA", "RF_HFE", "RF_KFE"]
    assert r.contact_frame_names == ["LF_FOOT", "LH_FOOT", "RF_FOOT", "RH_FOOT"]
    np.testing.assert_allclose(r.rotor_inertia, [0] * 6 + [0.1] * 12)
    assert all(m.effort_limit == 80.0 and m.velocity_limit == 7.5 and m.enable_velocity_limit for m in r.motors)
    # (-1, 0, 0) axes become RevoluteUnaligned, (1, 0, 0) RX
    kinds = dict(zip(r.joint_names, r.joint_type.tolist()))
    assert kinds["LF_HAA"] == M.JB_JOINT_RX and kinds["RF_HFE"] == M.JB_JOINT_RU and kinds["LH_HAA"] == M.JB_JOINT_RU
    lay = r.sensor_layout()
    assert lay["width"][0] == 66 and lay["ForceSensor"] == (6, 6, 4) and lay["EncoderSensor"] == (30, 2, 12)
    assert opt["stepper"]["controllerUpdatePeriod"] == 0.005 and opt["contacts"]["stiffness"] == 4.0e6


def test_atlas_contact_cleanup():
    r, _ = R.load_robot("atlas")
    assert (r.nq, r.nv, r.nmotors, r.njoints) == (37, 36, 30, 32)
    assert len(r.contact_frame_names) == 12 and sum(n.startswith("l_foot") for n in r.contact_frame_names) == 6
    assert r.contact_frame_names == sorted(r.contact_frame_names)


def test_compiled_tables_match_reference_data():
    """The shipped JSON tables are what the compiler produces from the reference's data files."""
    robot = M.build_robot_table(os.path.join(REF_ANYMAL, "anymal.urdf"), True)
    M.load_hardware_description_file(robot, os.path.join(REF_ANYMAL, "anymal_hardware.toml"))
    shipped, _ = R.load_robot("anymal")
    np.testing.assert_array_equal(robot.placement, shipped.placement)
    np.testing.assert_array_equal(robot.inertia, shipped.inertia)
    assert robot.contact_frame_names == shipped.contact_frame_names


def test_convex_hull_and_ground_height():
    pts = np.array([[0, 0], [1, 0], [1, 1], [0, 1], [0.5, 0.5], [0.5, 0.0]], dtype=float)
    assert sorted(R.convex_hull_2d_indices(pts).tolist()) == [0, 1, 2, 3]
    r, _ = R.load_robot("anymal")
    q = R.ground_base_height(r, r.neutral())
    z = [p.p[2] for p in R.frame_placements(r, q, r.contact_frame_names).values()]
    np.testing.assert_allclose(min(z), 0.0, atol=1e-15)


def test_option_validation():
    opt = M.default_engine_options()
    opt["stepper"]["dtMax"] = 0.5
    with pytest.raises(ValueError):
        M.validate_options(opt)
    opt = M.default_engine_options()
    opt["stepper"]["controllerUpdatePeriod"] = 0.003
    opt["stepper"]["sensorsUpdatePeriod"] = 0.005
    with pytest.raises(ValueError):
        M.validate_options(opt)


def test_robot_model_options_like_the_reference_tests():
    """`jiminy.Robot.get_model_options / set_model_options` over the tables: the flexibility API test
    (unit_py/test_simple_pendulum.py:815-842), the joint-limit options of unit_py/test_dense_pole.py:38-43, backlash from
    the motor options (test_simple_pendulum.py:276-284), theoretical <-> extended state maps."""
    import os
    import numpy as np
    from jiminy_b200 import model as M
    from conftest import DATA
    th = M.build_robot_table(os.path.join(DATA, "simple_pendulum.urdf"), False)
    M.attach_motor(th, "PendulumJoint", "PendulumJoint", enableVelocityLimit=False, enableEffortLimit=False,
                   enableArmature=True, armature=0.1, enableBacklash=True, backlash=0.4)
    robot = M.Robot(th)
    assert not robot.is_flexibility_enabled and robot.backlash_joint_names == ["PendulumJointBacklash"]
    opts = robot.get_model_options()
    assert opts["dynamics"]["enableFlexibility"] is True and opts["joints"]["positionLimitFromUrdf"] is True
    opts["dynamics"]["flexibilityConfig"] = [{"frameName": "PendulumJoint", "stiffness": np.ones(3), "damping": np.ones(3),
                                              "inertia": np.ones(3)}]
    opts["joints"]["positionLimitFromUrdf"] = False
    opts["joints"]["positionLimitLower"], opts["joints"]["positionLimitUpper"] = [-0.002], [0.002]
    robot.set_model_options(opts)
    ext = robot.extended
    assert robot.flexibility_joint_indices == [1]
    assert ext.joint_names == ["universe", "PendulumJointFlexibility", "PendulumJoint", "PendulumJointBacklash"]
    iq = ext.idx_q[ext.joint_index("PendulumJoint")]
    assert (ext.q_lower[iq], ext.q_upper[iq]) == (-0.002, 0.002) and (ext.q_lower[iq + 1], ext.q_upper[iq + 1]) == (-0.2, 0.2)
    assert th.njoints == 2 and robot.theoretical is th                      # the theoretical model is left alone
    qe = robot.get_extended_position_from_theoretical(np.array([0.3]))
    np.testing.assert_allclose(qe, [0.0, 0.0, 0.0, 1.0, 0.3, 0.0])
    np.testing.assert_allclose(robot.get_theoretical_position_from_extended(qe), [0.3])
    np.testing.assert_allclose(robot.get_extended_velocity_from_theoretical(np.array([2.0])), [0.0, 0.0, 0.0, 2.0, 0.0])
    bad = robot.get_model_options()
    bad["joints"]["positionLimitLower"] = [0.0, 1.0]
    with pytest.raises(ValueError):
        robot.set_model_options(bad)
    assert robot.flexibility_joint_indices == [1]                            # a refused update changes nothing
    opts["dynamics"]["enableFlexibility"] = False
    robot.set_model_options(opts)
    assert not robot.is_flexibility_enabled and robot.extended.joint_names == ["universe", "PendulumJoint", "PendulumJointBacklash"]

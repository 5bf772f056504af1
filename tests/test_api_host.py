"""Host-side logic of the drop-in layer (no GPU): model container, URDF
loader, limit selection, problem description, error behaviour."""

import os

import numpy as np
import pytest
import torch

import pink_b200
from pink_b200 import ComTask, FrameTask, PostureTask, RelativeFrameTask, _cabi
from pink_b200.exceptions import FrameNotFound, PinkError, TargetNotSet, TaskDefinitionError
from pink_b200.limits import ConfigurationLimit, VelocityLimit
from pink_b200.model import JointModelFreeFlyer, SE3, load_urdf, model_from_urdf_string
from pink_b200.solve_ik import describe_problem
from pink_b200.utils import VectorSpace, custom_configuration_vector, get_joint_idx, get_root_joint_dim
from tests import helpers

REF_ROBOTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_robots")


def test_ur5_model_dimensions_and_zero_pose():
    robot, model, table = helpers.load("ur5_description")
    assert (model.nq, model.nv, table.njoints) == (6, 6, 6)
    assert model.existFrame("tool0") and model.getFrameId("nope") == len(model.frames)
    assert get_root_joint_dim(model) == (0, 0)
    assert model.joints[0].idx_q == -1  # universe
    from oracle import kinematics as okin

    R, p = okin.frame_placement(table, okin.forward_kinematics(table, np.zeros(6)), table.frame_names.index("tool0"))
    # known zero pose of the UR5 (sum of the DH offsets)
    np.testing.assert_allclose(p, [0.81725, 0.19145, -0.005491], atol=1e-12)


def test_free_flyer_models_follow_pinocchio_conventions():
    for name, nj in [("draco3_description", 27), ("g1_description", 29)]:
        robot, model, table = helpers.load(name)
        assert (model.nq, model.nv) == (nj + 7, nj + 6)
        assert get_root_joint_dim(model) == (7, 6)
        assert model.names[1] == "root_joint" and model.joints[1].nq == 7
        np.testing.assert_array_equal(robot.q0[:7], [0, 0, 0, 0, 0, 0, 1])
        assert not model.hasConfigurationLimit()[3:7].any()
        # the floating base carries neither configuration nor velocity rows
        assert ConfigurationLimit(model).indices.min() >= 6
        assert VelocityLimit(model).indices.min() >= 6
        assert len(ConfigurationLimit(model).indices) == nj


@pytest.mark.parametrize("fname,nq", [("double_pendulum.urdf", 2), ("planar_2dof.urdf", 2), ("simple_pendulum.urdf", 1)])
def test_urdf_loader_on_the_reference_fixtures(fname, nq):
    robot = load_urdf(os.path.join(REF_ROBOTS, fname))
    assert robot.model.nq == nq == robot.model.nv
    table = robot.model.table()
    assert (table.parent == np.arange(-1, nq - 1)).all()
    # joints with lower == upper == 0 carry no configuration row (configuration_limit.py:50-56)
    lim = ConfigurationLimit(robot.model)
    expect = sum(1 for j in range(nq) if table.q_max[j] > table.q_min[j] + 1e-10)
    assert len(lim.indices) == expect


def test_urdf_fixed_joints_and_inertias_are_merged():
    xml = """<robot name="t">
      <link name="a"><inertial><mass value="1"/><origin xyz="0 0 0"/></inertial></link>
      <link name="b"><inertial><mass value="2"/><origin xyz="0 0 1"/></inertial></link>
      <link name="c"><inertial><mass value="2"/><origin xyz="1 0 0"/></inertial></link>
      <joint name="j1" type="revolute"><parent link="a"/><child link="b"/><origin xyz="0 0 1" rpy="0 0 0"/>
        <axis xyz="0 0 2"/><limit lower="-1" upper="1" velocity="2"/></joint>
      <joint name="f" type="fixed"><parent link="b"/><child link="c"/><origin xyz="0 1 0" rpy="0 0 1.5707963267948966"/></joint>
    </robot>"""
    model = model_from_urdf_string(xml)
    t = model.table()
    assert t.njoints == 1 and np.allclose(t.axis[0], [0, 0, 1])
    # body of j1 = links b and c: masses add, CoM is the weighted mean (c rotated by the fixed joint)
    assert t.mass[1] == 4.0
    np.testing.assert_allclose(t.com[1], (2 * np.array([0, 0, 1]) + 2 * np.array([0, 2, 0])) / 4, atol=1e-12)
    assert t.mass[0] == 0.0  # universe-attached inertia is ignored, as Pinocchio does
    assert model.existFrame("f") and model.existFrame("c")


def test_limit_selection_follows_the_reference():
    robot, model, table = helpers.load("ur5_description")
    cl, vl = ConfigurationLimit(model), VelocityLimit(model)
    assert list(cl.indices) == list(range(6)) and cl.projection_matrix.shape == (6, 6)
    lo, hi = cl.box_bounds()
    np.testing.assert_allclose(hi, table.q_max)
    # unlimited joints drop out
    model.upperPositionLimit = np.array([1e30, 1.0, 1.0, 0.0, 1.0, 1.0])
    model.lowerPositionLimit = np.array([-1e30, -1.0, -1.0, 0.0, -1.0, -1.0])
    assert list(ConfigurationLimit(model).indices) == [1, 2, 4, 5]
    v = np.array([1.0, 0.0, 1e25, 2.0, 2.0, 2.0])
    assert list(VelocityLimit(model, v).indices) == [0, 3, 4, 5]
    with pytest.raises(PinkError):
        VelocityLimit(model, np.ones(5))
    with pytest.raises(AssertionError):
        ConfigurationLimit(model, config_limit_gain=0.0)


def test_problem_description_layout():
    robot, model, table = helpers.load("ur5_description")
    B = 4
    ft = FrameTask("tool0", position_cost=[1.0, 2.0, 3.0], orientation_cost=0.5, lm_damping=0.2, gain=0.9)
    ft.set_target(torch.zeros(B, 3, 4))
    pt = PostureTask(cost=1e-3)
    pt.set_target(np.arange(6.0))
    prob, parts, descs = describe_problem(model, B, [ft, pt], 0.01, 1e-9,
                                          [ConfigurationLimit(model, 0.25), VelocityLimit(model)], True)
    assert prob.ntasks == 2 and prob.target_stride == 12 and len(parts) == 1
    t0, t1 = prob.tasks[0], prob.tasks[1]
    assert (t0.type, t0.target_shared, t0.target_offset) == (_cabi.PK_TASK_FRAME, 0, 0)
    np.testing.assert_allclose(list(t0.cost), [1, 2, 3, 0.5, 0.5, 0.5])
    assert abs(t0.gain - 0.9) < 1e-7 and abs(t0.lm_damping - 0.2) < 1e-7
    assert (t1.type, t1.target_shared, t1.target_offset) == (_cabi.PK_TASK_POSTURE, 1, 0)
    np.testing.assert_allclose(list(prob.shared[:6]), np.arange(6.0))
    assert abs(prob.cfg_gain - 0.25) < 1e-7
    np.testing.assert_allclose(list(prob.vel[:6]), table.v_max, rtol=1e-6)
    assert prob.cfg_hi[6] == float("inf") and prob.chk_lo[6] == -float("inf")
    np.testing.assert_allclose(list(prob.chk_hi[:6]), table.q_max + 1e-6, rtol=1e-6)
    # limits=[] => no rows at all
    prob2, _, _ = describe_problem(model, B, [pt], 0.01, 0.0, [], False)
    assert all(prob2.vel[i] == float("inf") for i in range(6)) and prob2.safety_break == 0


def test_task_error_behaviour():
    robot, model, table = helpers.load("g1_description")
    ft = FrameTask("pelvis", position_cost=1.0, orientation_cost=1.0)
    with pytest.raises(TargetNotSet):
        ft._pk_describe(model)
    ft.set_target(SE3())
    ft.frame = "does_not_exist"
    with pytest.raises(FrameNotFound):
        ft._pk_describe(model)
    with pytest.raises(AssertionError):
        FrameTask("pelvis", position_cost=-1.0, orientation_cost=1.0)
    bad = FrameTask("pelvis", position_cost=1.0, orientation_cost=1.0)
    bad.cost = 42.0
    with pytest.raises(TaskDefinitionError):
        bad.set_position_cost(1.0)
    for task in (PostureTask(cost=1.0), ComTask(cost=1.0), RelativeFrameTask("pelvis", "left_ankle_roll_link", 1.0, 1.0)):
        with pytest.raises(TargetNotSet):
            task._pk_describe(model)
    # targets are copied on set (frame_task.py:136)
    T = SE3(np.eye(3), np.array([0.0, 1.0, 0.0]))
    ok = FrameTask("pelvis", 1.0, 1.0)
    ok.set_target(T)
    T.translation[1] += 12.0
    assert abs(ok.transform_target_to_world.translation[1] - 1.0) < 1e-12
    # per-instance target count must match the batch
    ok.set_target(torch.zeros(3, 3, 4))
    with pytest.raises(PinkError):
        describe_problem(model, 5, [ok], 0.01, 0.0, [], False)
    assert "FrameTask(frame=pelvis" in repr(ok) and "PostureTask(cost=" in repr(PostureTask(cost=2.0))


def test_configuration_state_semantics():
    robot, model, table = helpers.load("ur5_description")
    q = np.linspace(-0.5, 0.5, 6)
    cfg = pink_b200.Configuration(model, robot.data, q)
    assert hasattr(model, "configuration_limit") and hasattr(model, "velocity_limit") and model.floating_base_velocity_limit is None
    assert isinstance(model.tangent, VectorSpace) and model.tangent.eye.shape == (6, 6)
    q[0] = 99.0
    assert cfg.q[0] != 99.0  # copied (configuration.py:109)
    with pytest.raises(ValueError):
        cfg.q[0] = 1.0  # read-only (tests/test_configuration.py:420-432)
    assert not cfg.batched and cfg.batch_size == 1
    cfgb = pink_b200.Configuration(model, robot.data, np.zeros((5, 6)))
    assert cfgb.batched and cfgb.batch_size == 5
    cfg.check_limits()
    bad = pink_b200.Configuration(model, robot.data, np.array([0, 0, 4.0, 0, 0, 0]))
    with pytest.raises(pink_b200.exceptions.NotWithinConfigurationLimits):
        bad.check_limits()
    bad.check_limits(safety_break=False)  # warns only
    with pytest.raises(ValueError):
        pink_b200.Configuration(model, robot.data, np.zeros(5))


def test_utils():
    robot, model, table = helpers.load("ur5_description")
    q = custom_configuration_vector(robot, elbow_joint=0.2)
    assert q[get_joint_idx(model, "elbow_joint")[0]] == 0.2
    with pytest.raises(pink_b200.exceptions.ConfigurationError):
        custom_configuration_vector(robot, elbow_joint=[0.1, 0.2])
    with pytest.raises(PinkError):
        get_joint_idx(model, "nope")


def test_se3_value_type():
    rng = np.random.default_rng(0)
    a, b = SE3.Random(rng), SE3.Random(rng)
    assert (a * a.inverse()).isApprox(SE3.Identity())
    assert a.actInv(b).isApprox(a.inverse() * b)
    np.testing.assert_allclose(a.action @ a.actionInverse, np.eye(6), atol=1e-12)
    np.testing.assert_allclose(np.asarray(a), a.homogeneous)
    assert SE3(a.homogeneous).isApprox(a) and SE3(a.as_3x4()).isApprox(a)


def test_sphere_collision_model_from_urdf_and_srdf(tmp_path):
    """Sphere-decomposed URDF -> SphereCollisionModel; process_collision_pairs with an SRDF
    (pink/utils.py:116-142, tests/test_self_collision_barrier.py:26-43)."""
    from pink_b200 import SphereCollisionModel
    from pink_b200.barriers import SelfCollisionBarrier
    from pink_b200.utils import process_collision_pairs

    urdf = """
    <robot name="spheres">
      <link name="base"><collision><origin xyz="0 0 0.1"/><geometry><sphere radius="0.1"/></geometry></collision></link>
      <link name="l1">
        <collision><origin xyz="0.1 0 0"/><geometry><sphere radius="0.05"/></geometry></collision>
        <collision><origin xyz="0.2 0 0"/><geometry><sphere radius="0.04"/></geometry></collision>
        <collision><geometry><box size="1 1 1"/></geometry></collision>
      </link>
      <link name="l2"><collision><origin xyz="0 0.1 0"/><geometry><sphere radius="0.03"/></geometry></collision></link>
      <joint name="j1" type="revolute"><parent link="base"/><child link="l1"/><origin xyz="0 0 0.3"/>
        <axis xyz="0 0 1"/><limit lower="-1" upper="1" velocity="2"/></joint>
      <joint name="j2" type="revolute"><parent link="l1"/><child link="l2"/><origin xyz="0.3 0 0" rpy="0 0 1.5707963"/>
        <axis xyz="0 1 0"/><limit lower="-1" upper="1" velocity="2"/></joint>
    </robot>"""
    model = model_from_urdf_string(urdf)
    cm = SphereCollisionModel.from_urdf_string(model, urdf)
    assert cm.names == ["base_0", "l1_0", "l1_1", "l2_0"] and cm.radii == [0.1, 0.05, 0.04, 0.03]
    assert cm.links == ["base", "l1", "l1", "l2"]
    # centres in the parent-joint frames (the base link hangs on the universe)
    table = model.table()
    f = table.frame_names.index("sphere:l1_1")
    np.testing.assert_allclose(table.frame_p[f], [0.2, 0.0, 0.0])
    srdf = tmp_path / "pairs.srdf"
    srdf.write_text('<robot name="spheres"><disable_collisions link1="base" link2="l1" reason="Adjacent"/></robot>')
    data = process_collision_pairs(model, cm, str(srdf))
    assert data.enable_contact and len(data.distanceResults) == 3
    names = {(cm.names[i], cm.names[j]) for i, j in cm.collisionPairs}
    # same-joint pairs are never added; base-l1 pairs are disabled by the SRDF
    assert names == {("base_0", "l2_0"), ("l1_0", "l2_0"), ("l1_1", "l2_0")}
    barrier = SelfCollisionBarrier(n_collision_pairs=2, d_min=0.01)
    prob, parts, _ = describe_problem(model, 4, [], 0.01, 1e-6, [], False, [barrier], None, cm)
    assert prob.nbarriers == 1 and prob.barriers[0].npairs == 3 and prob.n_pairs == 3 and prob.n_extra == 6
    from pink_b200.exceptions import InvalidCollisionPairs

    with pytest.raises(InvalidCollisionPairs):
        describe_problem(model, 4, [], 0.01, 1e-6, [], False, [SelfCollisionBarrier(n_collision_pairs=5)], None, cm)


def test_urdf_loader_rejects_malformed_trees():
    bad = {
        "undeclared link": '<robot name="r"><link name="a"/><joint name="j" type="revolute"><parent link="a"/>'
                           '<child link="zz"/><axis xyz="0 0 1"/></joint></robot>',
        "two roots": '<robot name="r"><link name="a"/><link name="b"/></robot>',
        "loop": '<robot name="r"><link name="a"/><link name="b"/><link name="c"/>'
                '<joint name="j1" type="revolute"><parent link="a"/><child link="c"/><axis xyz="0 0 1"/></joint>'
                '<joint name="j2" type="revolute"><parent link="b"/><child link="c"/><axis xyz="0 0 1"/></joint></robot>',
        "zero axis": '<robot name="r"><link name="a"/><link name="b"/><joint name="j" type="revolute">'
                     '<parent link="a"/><child link="b"/><axis xyz="0 0 0"/></joint></robot>',
    }
    for what, xml in bad.items():
        with pytest.raises(ValueError):
            model_from_urdf_string(xml)
    for jtype in ("planar", "floating"):
        with pytest.raises(NotImplementedError):
            model_from_urdf_string(f'<robot name="r"><link name="a"/><link name="b"/><joint name="j" type="{jtype}">'
                                   '<parent link="a"/><child link="b"/></joint></robot>')


@pytest.mark.parametrize("name,floating", [("ur5_description", False), ("draco3_description", True), ("g1_description", True)])
def test_model_flat_image_round_trip(name, floating):
    """Model.pack / Model.unpack (the payload of parallel.broadcast_model): numbers and names
    only, and the rebuilt model is the same model - tables, frame ids, limits, inertias."""
    from pink_b200.model import Model
    from pink_b200.robots import load_robot_description

    m = load_robot_description(name, root_joint=JointModelFreeFlyer() if floating else None).model
    floats, ints, text = m.pack()
    assert floats.dtype == np.float64 and ints.dtype == np.int64 and isinstance(text, bytes)
    m2 = Model.unpack(floats, ints, text)
    a, b = m.table(), m2.table()
    for key, val in vars(a).items():
        assert np.array_equal(np.asarray(val), np.asarray(getattr(b, key))), key
    assert [f.name for f in m.frames] == [f.name for f in m2.frames]
    assert m.names == m2.names and (m.nq, m.nv) == (m2.nq, m2.nv)
    np.testing.assert_array_equal(m.hasConfigurationLimit(), m2.hasConfigurationLimit())
    np.testing.assert_array_equal(m.velocityLimit, m2.velocityLimit)

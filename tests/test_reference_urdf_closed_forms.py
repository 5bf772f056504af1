"""Pins the URDF loader, forward kinematics and LOCAL frame Jacobians to files the REFERENCE
holds: the three robots it vendors under examples/robots (used by
examples/double_pendulum.py:28-36, planar_2dof_manipulability.py:35-43,
one_dof_configuration_limit.py:44-53), stored unmodified in tests/golden/reference_robots/.
Their kinematics has closed forms, written out below by hand from the URDF numbers -
independent of the oracle, of the model loader and of the kernels - so that all three are
tied to reference-held inputs:

* simple_pendulum: joint about x at the origin, tip 0.25 m up the body
      p = (0, -0.25 sin q, 0.25 cos q),  R = Rx(q)
* double_pendulum: joints about x at (0.025, 0, 0) and (0.0125, 0, 0.1), link3 0.2 m up link2
      p = (0.0375, -0.1 s1 - 0.2 s12, 0.1 c1 + 0.2 c12),  R = Rx(q1 + q2)
* planar_2dof: joints about z at (0.025, 0, 0) and (0.2, 0, 0), end effector 0.2 m along link2
      p = (0.025 + 0.2 c1 + 0.2 c12, 0.2 s1 + 0.2 s12, 0),  R = Rz(q1 + q2)

The LOCAL frame Jacobian (pink/configuration.py:233-235) follows from the same closed forms:
column i = [R^T (a_i x (p - p_i)); R^T a_i] with the joint axes / origins read off above.
Checked: the oracle (fp64), the host build of the kernels, and the CUDA library (-m gpu).
"""

import os

import numpy as np
import pytest

REF_ROBOTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_robots")


def Rx(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[1, 0, 0], [0, c, -s], [0, s, c]])


def Rz(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]])


def closed_form(name, q):
    """(frame name, R, p, J_local[6, nv]) at configuration q."""
    if name == "simple_pendulum.urdf":
        a = q[0]
        R = Rx(a)
        p = np.array([0.0, -0.25 * np.sin(a), 0.25 * np.cos(a)])
        axes, origins = [np.array([1.0, 0, 0])], [np.zeros(3)]
        frame = "tip"
    elif name == "double_pendulum.urdf":
        a, b = q
        R = Rx(a + b)
        p = np.array([0.0375, -0.1 * np.sin(a) - 0.2 * np.sin(a + b), 0.1 * np.cos(a) + 0.2 * np.cos(a + b)])
        axes = [np.array([1.0, 0, 0])] * 2
        origins = [np.array([0.025, 0, 0]), np.array([0.0375, -0.1 * np.sin(a), 0.1 * np.cos(a)])]
        frame = "link3"
    else:
        a, b = q
        R = Rz(a + b)
        p = np.array([0.025 + 0.2 * np.cos(a) + 0.2 * np.cos(a + b), 0.2 * np.sin(a) + 0.2 * np.sin(a + b), 0.0])
        axes = [np.array([0, 0, 1.0])] * 2
        origins = [np.array([0.025, 0, 0]), np.array([0.025 + 0.2 * np.cos(a), 0.2 * np.sin(a), 0.0])]
        frame = "end_effector"
    J = np.zeros((6, len(q)))
    for i, (ax, o) in enumerate(zip(axes, origins)):
        J[:3, i] = R.T @ np.cross(ax, p - o)
        J[3:, i] = R.T @ ax
    return frame, R, p, J


ROBOTS = [("simple_pendulum.urdf", 1), ("double_pendulum.urdf", 2), ("planar_2dof.urdf", 2)]


def _load(fname):
    from pink_b200.model import load_urdf

    robot = load_urdf(os.path.join(REF_ROBOTS, fname))
    return robot, robot.model.table()


def _configs(nq, n=40, seed=3):
    rng = np.random.default_rng(seed)
    return rng.uniform(-3.0, 3.0, size=(n, nq))


@pytest.mark.parametrize("fname,nq", ROBOTS)
def test_oracle_fk_and_local_jacobian_match_the_closed_forms(fname, nq):
    from oracle import kinematics as okin

    robot, table = _load(fname)
    q = _configs(nq)
    fk = okin.forward_kinematics(table, q)
    for i in range(q.shape[0]):
        frame, R, p, J = closed_form(fname, q[i])
        f = table.frame_names.index(frame)
        Ro, po = okin.frame_placement(table, fk, f)
        np.testing.assert_allclose(Ro[i], R, atol=1e-12)
        np.testing.assert_allclose(po[i], p, atol=1e-12)
        np.testing.assert_allclose(okin.frame_jacobian_local(table, fk, f)[i], J, atol=1e-12)


@pytest.mark.parametrize("fname,nq", ROBOTS)
def test_host_build_of_the_kernels_matches_the_closed_forms(fname, nq):
    from tests.hostsim import HostSim

    robot, table = _load(fname)
    hs = HostSim(robot.model)
    q = _configs(nq)
    oMf, _ = hs.forward_kinematics(q)
    frame = closed_form(fname, q[0])[0]
    f = table.frame_names.index(frame)
    Jh = hs.frame_jacobian(f, q)
    for i in range(q.shape[0]):
        _, R, p, J = closed_form(fname, q[i].astype(np.float32).astype(np.float64))
        np.testing.assert_allclose(oMf[i, f, :, :3], R, atol=2e-6)
        np.testing.assert_allclose(oMf[i, f, :, 3], p, atol=2e-6)
        np.testing.assert_allclose(Jh[i], J, atol=2e-6)


@pytest.mark.parametrize("fname,nq", ROBOTS)
def test_limits_read_from_the_reference_urdfs(fname, nq):
    robot, table = _load(fname)
    if fname == "simple_pendulum.urdf":  # <limit lower="0.0" upper="6.28" velocity="1.0"/>
        np.testing.assert_allclose([table.q_min[0], table.q_max[0], table.v_max[0]], [0.0, 6.28, 1.0])
    elif fname == "planar_2dof.urdf":  # <limit lower="-3.14159" upper="3.14159" velocity="2"/>
        np.testing.assert_allclose(table.q_min, [-3.14159] * 2)
        np.testing.assert_allclose(table.q_max, [3.14159] * 2)
        np.testing.assert_allclose(table.v_max, [2.0] * 2)
    else:  # lower = upper = 0, velocity = 0: no configuration and no velocity rows
        from pink_b200.limits import ConfigurationLimit, VelocityLimit

        assert len(ConfigurationLimit(robot.model).indices) == 0
        assert len(VelocityLimit(robot.model).indices) == 0


@pytest.mark.parametrize("fname,nq", ROBOTS)
def test_frame_task_error_and_jacobian_from_closed_forms(fname, nq):
    """FrameTask.compute_error / compute_jacobian (pink/tasks/frame_task.py:176-226) evaluated
    from the closed-form poses: e = log6(T_b^-1 T_t) and J = -Jlog6(T_t^-1 T_b) J_local, with
    log6 / Jlog6 from scipy's matrix logarithm and central differences - no oracle code."""
    from scipy.linalg import logm

    from oracle import tasks as otasks

    robot, table = _load(fname)
    rng = np.random.default_rng(5)
    q = rng.uniform(-1.0, 1.0, size=nq)
    qt = q + rng.normal(0, 0.2, size=nq)
    frame, R, p, J = closed_form(fname, q)
    _, Rt, pt, _ = closed_form(fname, qt)

    def log6(Ra, pa):
        T = np.eye(4)
        T[:3, :3], T[:3, 3] = Ra, pa
        Lg = np.real(logm(T))
        return np.array([Lg[0, 3], Lg[1, 3], Lg[2, 3], Lg[2, 1], Lg[0, 2], Lg[1, 0]])

    e_ref = log6(R.T @ Rt, R.T @ (pt - p))
    f = table.frame_names.index(frame)
    task = {"type": "frame", "frame": f, "cost": np.ones(6), "gain": 1.0, "lm_damping": 0.0,
            "target": (Rt[None], pt[None])}
    from oracle import kinematics as okin

    e, Jt = otasks.task_error_jacobian(table, q[None], okin.forward_kinematics(table, q[None]), task)
    np.testing.assert_allclose(e[0], e_ref, atol=1e-9)
    # de/dq by central differences of the closed form
    Jfd = np.zeros((6, nq))
    for k in range(nq):
        d = np.zeros(nq)
        d[k] = 1e-6
        _, Rp, pp, _ = closed_form(fname, q + d)
        _, Rm, pm, _ = closed_form(fname, q - d)
        Jfd[:, k] = (log6(Rp.T @ Rt, Rp.T @ (pt - pp)) - log6(Rm.T @ Rt, Rm.T @ (pt - pm))) / 2e-6
    np.testing.assert_allclose(Jt[0], Jfd, atol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("fname,nq", ROBOTS)
def test_cuda_library_matches_the_closed_forms(fname, nq):
    import torch

    from pink_b200.engine import get_engine

    robot, table = _load(fname)
    eng = get_engine(robot.model)
    q = _configs(nq).astype(np.float32)
    q_d = torch.as_tensor(q, device=eng.device)
    oMf, _ = eng.forward_kinematics(q_d)
    frame = closed_form(fname, q[0])[0]
    f = table.frame_names.index(frame)
    Jd = eng.frame_jacobian(f, q_d)
    torch.cuda.synchronize()
    oMf, Jd = oMf.cpu().numpy(), Jd.cpu().numpy()
    for i in range(q.shape[0]):
        _, R, p, J = closed_form(fname, q[i].astype(np.float64))
        np.testing.assert_allclose(oMf[i, f, :, :3], R, atol=2e-6)
        np.testing.assert_allclose(oMf[i, f, :, 3], p, atol=2e-6)
        np.testing.assert_allclose(Jd[i], J, atol=2e-6)

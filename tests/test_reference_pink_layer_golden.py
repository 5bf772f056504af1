"""Outputs of the REFERENCE's own Pink-layer Python, frozen under tests/golden/ref_pink_layer_*.npz
by scripts/make_reference_golden.py: the unmodified ``pink.build_ik`` / ``pink.solve_ik`` /
``Task.compute_error`` / ``compute_jacobian`` of /root/reference executed in the build container
over oracle-backed stand-ins for the two third-party modules it imports (oracle/refshim/README.md
says what that pins - task composition, weighting, LM rule, stacking order, limit / barrier /
equality rows, dq / dt - and what it leaves to the closed-form tests - the kinematic primitives and
the QP solver).

Checked here against those files: the oracle's restatement of the same layer (fp64, tight), the
host build of the kernels and, under ``-m gpu``, the CUDA library through the C ABI (fp32, the
tolerances of the parity suites).  Nothing in this file touches /root/reference or the shims."""

import os

import numpy as np
import pytest

from oracle import ik as oik
from oracle import kinematics as okin
from oracle import tasks as otk
from tests import helpers
from tests import ref_pink_layer_cases as cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    z = np.load(os.path.join(GOLDEN, f"ref_pink_layer_{name}.npz"))
    return {k: z[k] for k in z.files}


def _same(a, b, rtol=1e-10, atol=1e-12):
    a = np.zeros((0,)) if a is None else np.asarray(a)
    assert a.size == b.size, (a.shape, b.shape)
    if a.size:
        np.testing.assert_allclose(a.reshape(b.shape), b, rtol=rtol, atol=atol)


@pytest.mark.parametrize("name", cases.NAMES)
def test_oracle_assembly_equals_the_reference_build_ik(name):
    """(P, q, G, h, A, b) of every instance, row for row in the reference's stacking order."""
    case, gold = cases.build(name), _load(name)
    np.testing.assert_array_equal(case.q64, gold["inputs_q"])
    for i in range(case.B):
        tasks = [oik._slice_task(t, i) for t in case.otasks]
        cons = [oik._slice_task(t, i) for t in case.oconstraints]
        H, c, G, h, A, b = oik.assemble(case.table, case.q64[i], tasks, case.dt, case.damping,
                                        oik._slice_limits(case.olimits, i), case.obarriers, cons)
        scale = np.abs(gold["P"][i]).max()
        _same(H, gold["P"][i], atol=1e-12 * scale)
        _same(c, gold["q"][i], atol=1e-12 * max(1.0, np.abs(gold["q"][i]).max()))
        _same(G, gold["G"][i])
        _same(h, gold["h"][i])
        _same(A, gold["A"][i])
        _same(b, gold["b"][i])


@pytest.mark.parametrize("name", cases.NAMES)
def test_oracle_task_errors_and_jacobians_equal_the_reference_tasks(name):
    case, gold = cases.build(name), _load(name)
    for k, task in enumerate(case.otasks):
        for i in range(case.B):
            q = case.q64[i]
            fk = okin.forward_kinematics(case.table, q)
            e, J = otk.task_error_jacobian(case.table, q, fk, oik._slice_task(task, i))
            _same(e, gold[f"task{k}_e"][i])
            _same(J, gold[f"task{k}_J"][i])


@pytest.mark.parametrize("name", cases.NAMES)
def test_oracle_velocity_equals_the_reference_solve_ik(name):
    """Same QP solver on both sides (oracle/qp.py through the qpsolvers stand-in): any difference
    would come from the assembly or from ``Delta_q / dt``."""
    case, gold = cases.build(name), _load(name)
    for i in range(case.B):
        tasks = [oik._slice_task(t, i) for t in case.otasks]
        cons = [oik._slice_task(t, i) for t in case.oconstraints]
        v, status = oik.solve_ik(case.table, case.q64[i], tasks, case.dt, case.damping, oik._slice_limits(case.olimits, i),
                                 False, case.obarriers, cons)
        assert (status == 0) == bool(gold["found"][i])
        if gold["found"][i]:
            np.testing.assert_allclose(v, gold["v"][i], rtol=1e-9, atol=1e-10)


def _check_kernel(case, gold, v, st):
    ok = gold["found"] == 1
    assert (st[ok] == 0).all(), st
    assert ((st[~ok] & 1) != 0).all(), st
    assert helpers.within_tolerance(v[ok], gold["v"][ok], atol=1e-3, rtol=1e-2).all(), np.abs(v[ok] - gold["v"][ok]).max()
    assert helpers.within_tolerance(v[ok], gold["v"][ok], atol=5e-4, rtol=5e-3).mean() >= 0.8


def _describe(case):
    from pink_b200.solve_ik import describe_problem
    import torch

    prob, parts, _ = describe_problem(case.model, case.B, case.tasks, case.dt, case.damping, case.limits, case.safety_break,
                                      case.barriers, case.constraints, case.collision_model)
    targets = torch.cat([p.cpu().float() for p in parts], dim=1) if parts else None
    return prob, targets


@pytest.mark.parametrize("name", cases.NAMES)
def test_host_build_of_the_kernels_matches_the_reference_velocities(name):
    from tests.hostsim import HostSim

    case, gold = cases.build(name), _load(name)
    prob, targets = _describe(case)
    v, st = HostSim(case.model).solve_ik(prob, case.q32, None if targets is None else targets.numpy())
    _check_kernel(case, gold, v, st)


@pytest.mark.gpu
@pytest.mark.parametrize("name", cases.NAMES)
def test_cuda_library_matches_the_reference_velocities(name):
    """Through the C ABI (pk_solve_ik_batched via the engine)."""
    import torch

    from pink_b200.engine import get_engine

    case, gold = cases.build(name), _load(name)
    prob, targets = _describe(case)
    eng = get_engine(case.model)
    v, st = eng.solve_ik(prob, torch.as_tensor(case.q32, device=eng.device), None if targets is None else targets.to(eng.device))
    torch.cuda.synchronize()
    _check_kernel(case, gold, v.cpu().numpy(), st.cpu().numpy())


# ---- closed loops of two reference examples (tests/golden/ref_example_*.npz) ---------------------
def _example_robot(fname):
    from pink_b200.model import load_urdf

    return load_urdf(os.path.join(GOLDEN, "reference_robots", fname))


def _check_example(name, q, v):
    gold = np.load(os.path.join(GOLDEN, f"ref_example_{name}.npz"))
    # measured on the host build: 1.7e-4 rad over the 300 steps of the double pendulum (whose first
    # steps leave a singular pose at up to 400 rad/s), 2.4e-7 rad on the pendulum that runs into its limit
    assert np.abs(q - gold["q"]).max() <= (2e-3 if name == "double_pendulum" else 1e-5), np.abs(q - gold["q"]).max()
    assert helpers.within_tolerance(v, gold["v"], atol=5e-3, rtol=5e-3).all(), np.abs(v - gold["v"]).max()
    if name == "one_dof_configuration_limit":  # the example's point: stuck on the configuration limit
        assert abs(q[-1, 0]) <= 1e-6 and np.abs(v[-50:]).max() <= 1e-4


@pytest.mark.parametrize("name", sorted(cases.EXAMPLE_LOOPS))
def test_example_closed_loop_on_the_host_build_follows_the_reference_trajectory(name):
    """``examples/double_pendulum.py`` / ``examples/one_dof_configuration_limit.py`` as the reference's own
    code ran them (fixture) against the same loop through this package's unbatched API."""
    import pink_b200
    from tests.host_engine import HostEngine
    import pink_b200.configuration as cfgmod

    fname, steps = cases.EXAMPLE_LOOPS[name]
    cache = {}
    saved = cfgmod.get_engine
    cfgmod.get_engine = lambda model, device=None: cache.setdefault(id(model), HostEngine(model))
    try:
        q, v = cases.run_example_loop(name, pink_b200, _example_robot(fname), steps)
    finally:
        cfgmod.get_engine = saved
    _check_example(name, q, v)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(cases.EXAMPLE_LOOPS))
def test_example_closed_loop_on_the_gpu_follows_the_reference_trajectory(name):
    import pink_b200

    fname, steps = cases.EXAMPLE_LOOPS[name]
    q, v = cases.run_example_loop(name, pink_b200, _example_robot(fname), steps)
    _check_example(name, q, v)


def test_c_port_of_the_cpu_arm_equals_the_reference_on_the_benchmark_workload():
    """``bench.py --impl reference`` times oracle/c/pink_oracle.c: on the benchmark workload's generator
    and seed (B = 64) its velocities are those of the reference's own ``pink.solve_ik``."""
    from oracle import cport

    case, gold = cases.build("ur5_benchmark_workload"), _load("ur5_benchmark_workload")
    port = cport.CPort(case.table, case.otasks, case.dt, case.damping)
    R, p = case.otasks[0]["target"]
    targets = np.concatenate([R, p[:, :, None]], axis=2)[:, None]
    v, st = port.solve(case.q64, targets, threads=2)
    assert (st == 0).all() and gold["found"].all()
    np.testing.assert_allclose(v, gold["v"], rtol=1e-9, atol=1e-10)

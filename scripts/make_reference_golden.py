#!/usr/bin/env python3
"""Freeze outputs of the REFERENCE's own Pink-layer Python under tests/golden/ref_pink_layer_*.npz.

It imports the UNMODIFIED package ``pink`` of the reference, byte-compiled by ``build()`` into
``oracle/_ref/pink`` (oracle/ref_build.py), with the two name shims of ``oracle/refshim`` (``pinocchio``,
``qpsolvers``: oracle-backed stand-ins, see oracle/refshim/README.md) in front of it, because
the real third-party modules are neither installed nor installable here.  For every seeded
case it builds the reference's task / limit / barrier OBJECTS, then calls the reference's
``pink.build_ik`` and ``pink.solve_ik`` per instance and stores ``P, q, G, h, A, b``, the
velocity and every task's ``compute_error`` / ``compute_jacobian``.

    python scripts/make_reference_golden.py          # rewrites the fixtures (deterministic)
    python scripts/make_reference_golden.py --check  # re-runs the reference and compares with the committed files

``tests/test_reference_pink_layer_golden.py`` compares the oracle's own assembly (and the
kernels) with these files; nothing under tests/ imports the reference or the shims.

What the fixtures pin and what they do not: oracle/refshim/README.md.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = os.path.join(ROOT, "oracle", "_ref")
# order matters: the staged reference also has a package called `tests`
sys.path[:0] = [os.path.join(ROOT, "oracle", "refshim"), ROOT, REFERENCE]

import numpy as np  # noqa: E402
import pinocchio as pin  # noqa: E402  (the shim)
import pink  # noqa: E402  (the reference)
from pink.barriers import BodySphericalBarrier, PositionBarrier, SelfCollisionBarrier  # noqa: E402
from pink.limits import AccelerationLimit, ConfigurationLimit, FloatingBaseVelocityLimit, VelocityLimit  # noqa: E402
from pink.tasks import ComTask, DampingTask, FrameTask, JointCouplingTask, JointVelocityTask  # noqa: E402
from pink.tasks import LinearHolonomicTask, LowAccelerationTask  # noqa: E402
from pink.tasks import PostureTask, RelativeFrameTask  # noqa: E402

assert pink.__file__.startswith(REFERENCE), pink.__file__
assert pin.__file__.startswith(os.path.join(ROOT, "oracle", "refshim")), pin.__file__

from tests import ref_pink_layer_cases as cases  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
CHECK = "--check" in sys.argv


def reference_task(o, i, table, configuration):
    """Oracle task record ``o`` (tests/helpers.py, tests/extras.py) -> the reference's task object
    for instance ``i``."""
    kind = o["type"]
    cost = o.get("cost")
    gain, lm = o.get("gain", 1.0), o.get("lm_damping", 0.0)

    def se3(target):
        R, p = target
        R, p = np.asarray(R), np.asarray(p)
        return pin.SE3(R[i], p[i]) if R.ndim == 3 else pin.SE3(R, p)

    if kind == "frame":
        t = FrameTask(table.frame_names[o["frame"]], position_cost=np.asarray(cost[:3]), orientation_cost=np.asarray(cost[3:]),
                      lm_damping=lm, gain=gain)
        t.set_target(se3(o["target"]))
        return t
    if kind == "relative_frame":
        t = RelativeFrameTask(table.frame_names[o["frame"]], table.frame_names[o["root"]], position_cost=np.asarray(cost[:3]),
                              orientation_cost=np.asarray(cost[3:]), lm_damping=lm, gain=gain)
        t.set_target(se3(o["target"]))
        return t
    if kind == "posture":
        t = PostureTask(cost=cost, lm_damping=lm, gain=gain)
        t.set_target(np.asarray(o["target"], dtype=np.float64))
        return t
    if kind == "com":
        t = ComTask(cost=np.asarray(cost), lm_damping=lm, gain=gain)
        target = np.asarray(o["target"], dtype=np.float64)
        t.set_target(target[i] if target.ndim == 2 else target)
        return t
    if kind == "joint_velocity":
        target = np.asarray(o["target"], dtype=np.float64)
        target = target[i] if target.ndim == 2 else target
        if o.get("ref_class") == "damping":
            return DampingTask(cost=cost)
        if o.get("ref_class") == "joint_velocity":
            t = JointVelocityTask(cost=cost)
            t.set_target(target / o["ref_dt"], o["ref_dt"])
            return t
        # otherwise the record restates a LowAccelerationTask: e = -dt v_prev
        t = LowAccelerationTask(cost=cost)
        t.Delta_q_prev = -target
        return t
    if kind == "linear":
        A = np.asarray(o["A"], dtype=np.float64)
        if o.get("q0") is None:  # the JointCouplingTask of the scenario
            cols = np.nonzero(A[0])[0]
            names = [next(j.name for j in configuration.model.joints if j.idx_v == c and j.nv == 1) for c in cols]
            c0 = np.asarray(cost, dtype=np.float64).reshape(-1)
            return JointCouplingTask(names, [float(A[0, c]) for c in cols], float(c0[0]), configuration, lm_damping=lm, gain=gain)
        return LinearHolonomicTask(A, np.asarray(o["b"], dtype=np.float64), np.asarray(o["q0"], dtype=np.float64),
                                   cost=np.asarray(cost, dtype=np.float64), lm_damping=lm, gain=gain)
    raise ValueError(kind)


def reference_limits(olimits, i, model, table, dt):
    if olimits is None:
        return None  # the reference's default: model.configuration_limit, model.velocity_limit
    out = []
    for entry in olimits:
        if entry[0] == "configuration":
            out.append(ConfigurationLimit(model, config_limit_gain=entry[1]))
        elif entry[0] == "velocity":
            assert entry[1] is None
            out.append(VelocityLimit(model))
        elif entry[0] == "acceleration":
            lim = AccelerationLimit(model, np.asarray(entry[1], dtype=np.float64))
            dq_prev = np.asarray(entry[2], dtype=np.float64)
            dq_prev = dq_prev[i] if dq_prev.ndim == 2 else dq_prev
            lim.set_last_integration(dq_prev / dt, dt)
            out.append(lim)
        elif entry[0] == "floating_base":
            twist = np.asarray(entry[2], dtype=np.float64)
            out.append(FloatingBaseVelocityLimit(model, table.frame_names[entry[1]], twist[:3], twist[3:]))
        else:
            raise ValueError(entry[0])
    return out


def reference_barrier(o, table):
    if o["type"] == "position":
        return PositionBarrier(table.frame_names[o["frame"]], indices=list(o["indices"]), p_min=o["p_min"], p_max=o["p_max"],
                               gain=o["gain"], safe_displacement_gain=o["safe_displacement_gain"])
    if o["type"] == "body_spherical":
        a, b = o["frames"]
        return BodySphericalBarrier((table.frame_names[a], table.frame_names[b]), d_min=o["d_min"], gain=o["gain"],
                                    safe_displacement_gain=o["safe_displacement_gain"])
    if o["type"] == "self_collision":
        return SelfCollisionBarrier(n_collision_pairs=o["n_pairs"], gain=o["gain"], safe_displacement_gain=o["safe_displacement_gain"],
                                    d_min=o["d_min"])
    raise ValueError(o["type"])


def pad(rows, width=None):
    """Stack per-instance arrays (or None) into one array; None -> zero rows."""
    rows = [np.zeros((0,) + ((width,) if width else ())) if r is None else np.asarray(r, dtype=np.float64) for r in rows]
    return np.stack(rows)


def run_case(name):
    case = cases.build(name)
    model, table = case.model, case.table
    data = model.createData()
    out = {k: [] for k in ("P", "q", "G", "h", "A", "b", "v", "found")}
    task_e, task_J = {}, {}
    geometry = pin.GeometryModel(case.collision_model) if case.collision_model is not None else None
    for i in range(case.B):
        configuration = pink.Configuration(model, data, case.q64[i].copy(), collision_model=geometry)
        tasks = [reference_task(o, i, table, configuration) for o in case.otasks]
        limits = reference_limits(case.olimits, i, model, table, case.dt)
        barriers = [reference_barrier(o, table) for o in case.obarriers]
        constraints = [reference_task(o, i, table, configuration) for o in case.oconstraints]
        problem = pink.build_ik(configuration, tasks, case.dt, damping=case.damping, limits=limits,
                                barriers=barriers or None, constraints=constraints or None)
        for key, val in zip(("P", "q", "G", "h", "A", "b"), (problem.P, problem.q, problem.G, problem.h, problem.A, problem.b)):
            out[key].append(val)
        try:
            v = pink.solve_ik(configuration, tasks, case.dt, solver="quadprog", damping=case.damping, limits=limits,
                              barriers=barriers or None, constraints=constraints or None, safety_break=False)
            out["v"].append(v)
            out["found"].append(1)
        except pink.exceptions.NoSolutionFound:
            out["v"].append(np.zeros(model.nv))
            out["found"].append(0)
        for k, t in enumerate(tasks):
            task_e.setdefault(k, []).append(t.compute_error(configuration))
            task_J.setdefault(k, []).append(t.compute_jacobian(configuration))
    nv = model.nv
    arrays = {"inputs_q": case.q64, "P": pad(out["P"]), "q": pad(out["q"]), "G": pad(out["G"], nv), "h": pad(out["h"]),
              "A": pad(out["A"], nv), "b": pad(out["b"]), "v": pad(out["v"]), "found": np.array(out["found"])}
    for k in task_e:
        arrays[f"task{k}_e"] = pad(task_e[k])
        arrays[f"task{k}_J"] = pad(task_J[k])
    path = os.path.join(GOLDEN, f"ref_pink_layer_{name}.npz")
    if CHECK:  # compare with the committed fixture instead of rewriting it
        old = np.load(path)
        assert sorted(old.files) == sorted(arrays), (sorted(old.files), sorted(arrays))
        for k in arrays:
            np.testing.assert_allclose(np.asarray(arrays[k], dtype=np.float64), old[k], rtol=1e-12, atol=1e-14, err_msg=f"{name}:{k}")
        print(f"{name}: committed fixture reproduced")
        return
    np.savez_compressed(path, **arrays)
    print(f"{name}: {case.B} instances, nv {nv}, G rows {arrays['G'].shape[1]}, A rows {arrays['A'].shape[1]}, "
          f"solved {int(arrays['found'].sum())} -> {os.path.relpath(path, ROOT)} ({os.path.getsize(path) // 1024} KB)")


def run_example(name):
    """Closed loop of a reference example on the URDF the reference vendors for it."""
    fname, steps = cases.EXAMPLE_LOOPS[name]
    robot = pin.RobotWrapper(pin.pinocchio_like_limits(pin.load_urdf(os.path.join(GOLDEN, "reference_robots", fname)).model))
    q, v = cases.run_example_loop(name, pink, robot, steps)
    path = os.path.join(GOLDEN, f"ref_example_{name}.npz")
    if CHECK:
        old = np.load(path)
        np.testing.assert_allclose(q, old["q"], rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(v, old["v"], rtol=1e-12, atol=1e-13)
        print(f"example {name}: committed fixture reproduced")
        return
    np.savez_compressed(path, q=q, v=v)
    print(f"example {name}: {steps} steps, q from {q[0]} to {q[-1]} -> {os.path.relpath(path, ROOT)}")


if __name__ == "__main__":
    print(f"reference: pink {pink.__version__} from {os.path.dirname(pink.__file__)}")
    for name in cases.NAMES:
        run_case(name)
    for name in cases.EXAMPLE_LOOPS:
        run_example(name)

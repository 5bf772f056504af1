#!/usr/bin/env python3
"""Benchmark of the batched differential-IK hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

A "step" is one ``solve_ik`` pass over one batch of B = 65536 UR5 instances per
GPU (FrameTask(tool0) + PostureTask + default limits, examples/arm_ur5.py).
Prints ONE JSON line (rank 0).  See DESIGN.md section "Measurement".

How the K steps are timed (all of it holds for any K, the driver's K = 20 included):
the K launches of the fused kernel are submitted as CUDA-graph replays (one graph of
exactly K launches, or replays of a 512-launch graph plus a remainder graph for large
K), behind a short device-side spin so that the host has queued everything before the
start event fires; the region is bracketed by barrier + synchronize, repeated
``--regions`` times with an L2 flush in between, and the MEDIAN region is reported
(max over ranks).  ``roofline.timing`` says what ran.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "IK solves/sec (batch=65536 per GPU, UR5 6-DOF, FrameTask+PostureTask, default limits)"
UNIT = "IK steps/s"
BYTES_PER_STEP = 96  # q 24 B + frame target 48 B read, v 24 B written (BASELINE.md section 4)
L2_BYTES = 126 * 1024 * 1024
GRAPH_CHUNK = 512    # launches per captured graph when K is larger than this
DUMP_LIMIT = 64_000_000  # bytes --dump-outputs may write in all, .npy headers included


def dump_outputs(out_dir, arrays):
    """``--dump-outputs``: every array of ``arrays`` (name -> [B, ...] over the same B instances)
    as ``out_dir/<name>.npy``, float64 kept, anything else as float32.  When they would exceed
    DUMP_LIMIT, every array keeps the same fixed, seeded sample of instances (ascending), and the
    instance indices are written as ``instance.npy``."""
    arrays = {k: a if a.dtype == np.float64 else a.astype(np.float32) for k, a in arrays.items()}
    budget = DUMP_LIMIT - 256 * (len(arrays) + 1)  # room for the .npy headers (128 bytes each here)
    total = sum(a.nbytes for a in arrays.values())
    if total > budget:
        B = next(iter(arrays.values())).shape[0]
        n = budget * B // (total + 8 * B)  # rows that fit together with their float64 index
        rows = np.sort(np.random.default_rng(0).choice(B, size=n, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["instance"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def committed_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu --set full
    capture (profiles/traffic.json names the capture and its conditions); None when absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            d = json.load(f)
        return d["dram_bytes_per_launch"], d.get("capture")
    except (OSError, KeyError, ValueError):
        return None, None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def host_topology():
    """(logical CPUs this process may run on, physical cores among them)."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except AttributeError:
        cpus = list(range(os.cpu_count() or 1))
    cores = set()
    for c in cpus:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as fh:
                cores.add(fh.read().strip())
        except OSError:
            cores.add(str(c))
    return len(cpus), len(cores)


def cpu_quota():
    """CPUs' worth of run time the container may use per period (cgroup CFS quota), or None.
    On the GPU boxes of this pool the container sees 128 logical CPUs but `cpu.max` is
    `1600000 100000`: 16 CPUs sustained.  More runnable threads than that burn the period's
    budget in a burst and are then throttled for tens of milliseconds (measured with
    scripts/cpu_pool_diag.py: 128 threads alternate 2.6 ms steps with 45-85 ms stalls)."""
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:  # cgroup v2
            quota, period = fh.read().split()[:2]
        if quota != "max":
            return float(quota) / float(period)
    except (OSError, ValueError):
        pass
    try:  # cgroup v1
        with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as fh:
            quota = float(fh.read())
        with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as fh:
            period = float(fh.read())
        if quota > 0:
            return quota / period
    except (OSError, ValueError):
        pass
    return None


def cpu_threads():
    """(threads the CPU arm runs on, logical CPUs, physical cores, quota): every CPU the process may
    use, capped by the CFS quota (running more threads than the quota allows only adds
    throttling stalls)."""
    logical, physical = host_topology()
    quota = cpu_quota()
    threads = logical if quota is None else max(1, min(logical, int(quota)))
    return threads, logical, physical, quota


def bind_to_gpu_numa_node(index: int):
    """Run this process (and therefore first-touch its pinned buffers) on the NUMA node the
    GPU hangs off: host<->device DMA that crosses the socket interconnect runs well below
    the PCIe rate.  Returns a short description for the JSON line."""
    try:
        import pynvml

        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:  # 00000000:17:00.0 -> 0000:17:00.0
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as fh:
            node = int(fh.read().strip())
        if node < 0:
            return "numa node unknown (single node or virtualised)"
        with open(f"/sys/devices/system/node/node{node}/cpulist") as fh:
            spec = fh.read().strip()
        cpus = set()
        for part in spec.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if not allowed:
            return f"numa node {node}: no allowed CPU there"
        os.sched_setaffinity(0, allowed)
        return f"numa node {node} ({len(allowed)} CPUs)"
    except Exception as exc:  # best effort; never fail the bench on a topology quirk
        return f"not bound ({type(exc).__name__})"


# ---------------------------------------------------------------------------
# CPU arm: the oracle's C port of the reference path, all host cores
# ---------------------------------------------------------------------------


class CpuArm:
    """fp64 CPU implementation of the same step (oracle/c/pink_oracle.c: dense H,
    Goldfarb-Idnani QP with Givens updates, persistent pinned pthread pool).  Pink +
    Pinocchio + quadprog cannot be installed offline, so this port stands in for them."""

    def __init__(self, batch, seed=20260922):
        from oracle import cport
        from oracle import kinematics as okin
        from pink_b200 import workloads as wl
        from pink_b200.robots import load_robot_description

        robot = load_robot_description("ur5_description")
        table = robot.model.table()
        f = table.frame_names.index("tool0")
        rng = np.random.default_rng(seed)
        q = wl.sample_configurations(table, batch, rng)
        qt = wl.perturb_configurations(table, q, rng)
        R, p = okin.frame_placement(table, okin.forward_kinematics(table, qt), f)
        self.T = np.ascontiguousarray(
            np.concatenate([R, p[:, :, None]], axis=2).astype(np.float32).astype(np.float64)[:, None])
        self.q = np.ascontiguousarray(q.astype(np.float32).astype(np.float64))
        tasks = [
            {"type": "frame", "frame": f, "cost": np.ones(6), "gain": 1.0, "lm_damping": 1.0},
            {"type": "posture", "cost": 1e-3, "gain": 1.0, "lm_damping": 0.0,
             "target": wl.ur5_posture_reference(robot.model)},
        ]
        self.port = cport.CPort(table, tasks, wl.UR5_DT, wl.UR5_DAMPING)
        self.batch = batch
        self.table, self.model, self.wl = table, robot.model, wl

    def step(self, threads):
        t0 = time.perf_counter()
        v, st = self.port.solve(self.q, self.T, threads=threads, reuse_outputs=True)
        return time.perf_counter() - t0, v, st

    def python_port_rate(self, n=200):
        """The numpy per-instance loop (structure of the reference's Python path), 1 core."""
        from oracle import ik as oik

        f = self.table.frame_names.index("tool0")
        tasks = [
            {"type": "frame", "frame": f, "cost": np.ones(6), "gain": 1.0, "lm_damping": 1.0,
             "target": (self.T[:n, 0, :, :3], self.T[:n, 0, :, 3])},
            {"type": "posture", "cost": 1e-3, "gain": 1.0, "lm_damping": 0.0,
             "target": self.wl.ur5_posture_reference(self.model)},
        ]
        t0 = time.perf_counter()
        oik.solve_ik_batch(self.table, self.q[:n], tasks, self.wl.UR5_DT, self.wl.UR5_DAMPING)
        return n / (time.perf_counter() - t0)


def cpu_scaling(arm, passes, threads, cores_available):
    """All-thread and one-thread rates of the C port and the parallel efficiency against
    `cores available x one core` (available = physical cores, capped by the CFS quota)."""
    arm.step(threads)  # warm-up: pool creation, page faults
    arm.step(threads)
    wall = sum(arm.step(threads)[0] for _ in range(passes))
    one = min(arm.step(1)[0] for _ in range(2))
    value = arm.batch * passes / wall
    one_core = arm.batch / one
    return value, one_core, value / (one_core * cores_available)


def cpu_baseline_fields(value, one_core, threads, logical, physical, quota):
    avail = physical if quota is None else min(physical, quota)
    return {
        "value": value, "unit": UNIT, "cores": threads, "logical_cpus_visible": logical, "physical_cores_visible": physical,
        "cfs_quota_cpus": quota, "kind": "port", "one_core": one_core,
        "parallel_efficiency": value / (one_core * avail),
    }


def cpu_baseline_block(batch, passes=20):
    threads, logical, physical, quota = cpu_threads()
    arm = CpuArm(batch)
    avail = physical if quota is None else min(physical, quota)
    value, one_core, _ = cpu_scaling(arm, passes, threads, avail)
    out = cpu_baseline_fields(value, one_core, threads, logical, physical, quota)
    out["sample"] = (f"{passes} passes over the same {batch}-instance UR5 workload, fp64 C port of the reference path "
                     f"(dense H, Goldfarb-Idnani QP), persistent pool of {threads} pinned threads (futex wake-up, guided "
                     "chunks); thread count = CPUs the container may use (cgroup cpu.max); "
                     "Pink/Pinocchio/quadprog are not installable offline")
    out["python_loop_one_core"] = arm.python_port_rate()
    return out


def run_reference_arm(args):
    """``--impl reference``: the reference's CPU path on all host cores (the
    oracle's C port; the real stack cannot be installed offline)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads, logical, physical, quota = cpu_threads()
    arm = CpuArm(args.batch)
    for _ in range(max(args.warmup, 2)):
        arm.step(threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _, v, st = arm.step(threads)
    wall = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"v": v, "status": st})
    value = args.batch * args.steps / wall
    one = min(arm.step(1)[0] for _ in range(2))
    one_core = args.batch / one
    sample = (f"every step = the full {args.batch}-instance workload, fp64 C port of the reference path "
              f"(oracle/c/pink_oracle.c), persistent pool of {threads} pinned threads = the CPUs the container may use "
              f"({logical} logical CPUs visible, cgroup quota {quota})")
    cpu_block = cpu_baseline_fields(value, one_core, threads, logical, physical, quota)
    cpu_block["sample"] = sample
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": cpu_block,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args):
    """Identical for both arms (the driver compares them); the GPU arm's cache policy
    lives in ``roofline.l2``."""
    return {
        "workload": "UR5 6-DOF (hand-authored URDF), FrameTask(tool0, 1, 1, lm_damping=1) + PostureTask(1e-3), "
                    "ConfigurationLimit + VelocityLimit, dt=1/200, damping=1e-12 (examples/arm_ur5.py)",
        "batch_per_gpu": args.batch,
        "targets": "reachable: FK(q + N(0, 0.3^2)) clipped to limits; seed 20260922",
    }


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------


class ClockSampler:
    """Samples SM clocks / throttle reasons while the timed regions run.  In-process NVML
    (no subprocess per sample: an `nvidia-smi` spawned every 100 ms competes with the
    thread that issues the launches); falls back to nvidia-smi when NVML is missing."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, period: float = 0.02):
        self.index, self.period = index, period
        self.sm, self.mx, self.reasons = [], [], set()
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)
        self.source = "nvml"
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None
            self.source = "nvidia-smi"
            self.period = 0.25

    def _sample_nvml(self):
        nv = self._nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
        self.mx.append(self._max)
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for bit, name in self.REASONS.items():
            if mask & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(
            ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits"],
            capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
            s = [x.strip() for x in out.split(",")]
            self.sm.append(float(s[0]))
            self.mx.append(float(s[1]))
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[3:7]):
                if val.lower().startswith("active"):
                    self.reasons.add(name)

    def _run(self):
        while not self._stop.is_set():
            try:
                (self._sample_nvml if self._nv else self._sample_smi)()
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=6)

    def summary(self):
        return {
            "sm_mhz": float(np.median(self.sm)) if self.sm else None,
            "sm_max_mhz": float(max(self.mx)) if self.mx else None,
            "reasons": sorted(self.reasons),
            "samples": len(self.sm),
            "source": self.source,
        }


class GraphedSteps:
    """K launches of `step(k)` as CUDA-graph replays: one graph of exactly K launches when
    K <= GRAPH_CHUNK, else replays of a GRAPH_CHUNK-launch graph plus a remainder graph."""

    def __init__(self, torch, device, step, n_steps, chunk=GRAPH_CHUNK, end=None):
        self.torch, self.device, self.n = torch, device, n_steps
        self.end = end  # called at the end of every captured graph (joins side streams)
        self.full, self.rem = divmod(n_steps, chunk) if n_steps > chunk else (0, n_steps)
        self.chunk = chunk
        self.g_full = self._capture(step, 0, chunk) if self.full else None
        self.g_rem = self._capture(step, self.full * chunk, self.rem) if self.rem else None

    def _capture(self, step, k0, n):
        torch = self.torch
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            # thread-local capture mode: the NCCL watchdog thread of a multi-rank run may
            # issue CUDA calls (event queries) while this thread is capturing
            with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
                for k in range(n):
                    step(k0 + k)
                if self.end is not None:
                    self.end()
        torch.cuda.current_stream(self.device).wait_stream(side)
        return g

    def run(self):
        for _ in range(self.full):
            self.g_full.replay()
        if self.g_rem is not None:
            self.g_rem.replay()

    def describe(self):
        if self.full:
            return (f"{self.full} replays of a {self.chunk}-launch CUDA graph"
                    + (f" + one {self.rem}-launch graph" if self.rem else ""))
        return f"one replay of a {self.rem}-launch CUDA graph"


def kkt_selfcheck(ik, eng, q, targets, v, status, sample=512):
    """fp64 optimality certificate of the fp32 velocities on the QP the library itself
    exports (pk_build_ik_batched / pk_constraint_rows_batched) for the first `sample`
    instances: stationarity relative to the gradient's rounding scale, worst violation of
    the box and of the dense rows.  A self-consistency check of the solver inside the run;
    parity against the oracle is `pytest -m gpu`."""
    n = min(sample, q.shape[0])
    qs, ts = q[:n].contiguous(), targets[:n].contiguous()
    H, c, _ = eng.build_ik(ik.prob, qs, ts)
    G, hG, E, f, lo, hi = eng.constraint_rows(ik.prob, qs, ts)
    import torch

    torch.cuda.synchronize()
    ok = (status[:n] == 0).cpu().numpy()
    H, c = H.double().cpu().numpy()[ok], c.double().cpu().numpy()[ok]
    lo, hi = lo.double().cpu().numpy()[ok], hi.double().cpu().numpy()[ok]
    G, hG = G.double().cpu().numpy()[ok], hG.double().cpu().numpy()[ok]
    x = v[:n].double().cpu().numpy()[ok] * float(ik.prob.dt)
    g = np.einsum("bij,bj->bi", H, x) + c
    rows = np.abs(G).sum(axis=2) > 0  # unused dense rows are zero
    slack = hG - np.einsum("brj,bj->br", G, x)
    dense_viol = float(np.where(rows, np.maximum(-slack, 0.0), 0.0).max()) if rows.any() else 0.0
    # multipliers of active dense rows by least squares on the stationarity equation
    tol = 1e-9 + 1e-6 * np.abs(x) + 3e-7
    at_hi, at_lo = x >= hi - tol, x <= lo + tol
    resid = np.array(g)
    if rows.any():
        for b in range(x.shape[0]):
            act = rows[b] & (slack[b] <= 1e-6 * (1.0 + np.abs(hG[b])))
            if act.any():
                free = ~(at_hi[b] | at_lo[b])
                if free.any():
                    lam, *_ = np.linalg.lstsq(G[b][act][:, free].T, -g[b][free], rcond=None)
                    lam = np.maximum(lam, 0.0)
                    resid[b] = g[b] + G[b][act].T @ lam
    viol = np.abs(resid)
    viol = np.where(at_hi & (resid <= 0), 0.0, viol)
    viol = np.where(at_lo & (resid >= 0), 0.0, viol)
    scale = np.einsum("bij,bj->bi", np.abs(H), np.abs(x)).max(axis=1) + np.abs(c).max(axis=1)
    ratio = viol.max(axis=1) / scale
    return {
        "instances": int(ok.sum()), "stationarity_over_scale_p999": float(np.quantile(ratio, 0.999)),
        "stationarity_over_scale_max": float(ratio.max()),
        "box_violation_max": float(np.maximum(np.maximum(x - hi, lo - x), 0.0).max()),
        "dense_row_violation_max": dense_viol,
        "nonzero_status": int((~ok).sum()),
    }


def humanoid_configs(torch, device, peak, regions=5, steps=5):
    """BASELINE configs 3 and 4 (without and with the self-collision barrier): ms per step
    (median of `regions` timed regions of `steps` graph-replayed launches), algorithmic
    GB/s, status counts and the in-run KKT self-check."""
    from pink_b200 import workloads
    from pink_b200.engine import get_engine

    out = []
    for label, name, barrier in [("config 3: Draco3-class 27 joints + free-flyer, 4 FrameTasks + PostureTask", "draco3_description", False),
                                 ("config 4 without the barrier: G1-class 29 joints + free-flyer, ComTask + 5 FrameTasks + PostureTask", "g1_description", False),
                                 ("config 4: G1-class + sphere self-collision barrier (36 pairs, 8 closest)", "g1_description", True)]:
        ik, q_d, targets, model = workloads.humanoid_problem(name, device, with_barrier=barrier)
        B = q_d.shape[0]
        v = torch.empty((B, model.nv), dtype=torch.float32, device=device)
        st = torch.empty((B,), dtype=torch.int32, device=device)
        for _ in range(3):
            ik.solve(q_d, targets, v, st)
        torch.cuda.synchronize()
        graphed = GraphedSteps(torch, device, lambda k: ik.solve(q_d, targets, v, st), steps)
        graphed.run()
        torch.cuda.synchronize()
        times = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(regions):
            torch.cuda.synchronize()
            torch.cuda._sleep(200000)
            e0.record()
            graphed.run()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / steps)
        ms = float(np.median(times))
        nbytes = workloads.HUMANOID_BYTES_PER_STEP[name]
        ach = B * nbytes / (ms * 1e-3) / 1e9
        counts = {int(k): int(c) for k, c in zip(*np.unique(st.cpu().numpy(), return_counts=True))}
        out.append({
            "config": label, "robot": name + " (synthetic model of that class)", "batch": B, "nv": model.nv,
            "ms_per_step": ms, "ik_steps_per_s": B / (ms * 1e-3), "algorithmic_bytes_per_step": nbytes,
            "hbm_gbs_algorithmic": ach, "hbm_frac": ach / peak, "status_counts": counts,
            "kkt_selfcheck": kkt_selfcheck(ik, get_engine(model, device), q_d, targets, v, st),
            "timing": f"median of {regions} regions of {steps} graph-replayed launches",
        })
        del graphed, ik
    return out


def gather_variants(torch, dist, device, world, B, NBUF, step, vs, args, timed_regions, ik, qs, ts, ss):
    """solve + all-gather of v on every rank (the one data-path collective north_star names),
    three schedules, all submitted as CUDA-graph replays like the headline (median of regions,
    max over ranks):
    `serial`     - ncclAllGather on the solve stream after every step;
    `overlapped` - the gather of step k on a side stream (double-buffered output) while step
                   k + 1 solves; the region ends when the last gather has landed;
    `fused`      - the solve kernel stores its rows into every peer's gather buffer itself
                   (NVLink peer memory, pink_b200.parallel.PeerGather) and publishes "gather
                   k complete"; the wait for the peers' rows runs on a side stream, a
                   produced / released count per rank keeps a fast rank from overwriting a slot
                   a slower one still reads;
    `fused_wait_inline` - the same with the wait on the compute stream;
    `fused_two_in_flight` - two such sequences alternating over two compute streams (two
                   independent batches in flight, as `roofline.two_batches_in_flight_ms_per_step`
                   for the solve alone)."""
    from pink_b200 import parallel

    gathered = [torch.empty((world * B, 6), dtype=torch.float32, device=device) for _ in range(2)]
    peer = parallel.PeerGather(B, 6, device, n_buffers=2)

    def serial(k):
        step(k)
        dist.all_gather_into_tensor(gathered[0], vs[k % NBUF])

    class Overlapped:
        def __init__(self):
            self.side = torch.cuda.Stream(device)

        def __call__(self, k):
            cur = torch.cuda.current_stream(device)
            step(k)
            self.side.wait_stream(cur)
            with torch.cuda.stream(self.side):
                dist.all_gather_into_tensor(gathered[k % 2], vs[k % NBUF])

        def end(self):
            torch.cuda.current_stream(device).wait_stream(self.side)

    class Fused:
        """solve (+ fused gather) on the compute stream, the matching wait / release on a side
        stream: the next solve overlaps this one's NVLink drain and flag round trip"""

        def __init__(self):
            self.side = torch.cuda.Stream(device)

        def __call__(self, k):
            i = k % NBUF
            cur = torch.cuda.current_stream(device)
            peer.solve(ik, qs[i], ts[i], ss[i], vs[i], wait=False)
            self.side.wait_stream(cur)
            with torch.cuda.stream(self.side):
                peer.wait()

        def end(self):
            torch.cuda.current_stream(device).wait_stream(self.side)

    class FusedSerial:
        """the same with the wait on the compute stream (what PeerGather.solve does by default)"""

        def __call__(self, k):
            i = k % NBUF
            peer.solve(ik, qs[i], ts[i], ss[i], vs[i])

    class FusedTwoInFlight:
        """two gather sequences in flight: even steps on one compute stream with one PeerGather,
        odd steps on a second stream with a second PeerGather (own buffers and counters), each
        with its wait on its own side stream.  A one-wave kernel emits its peer stores as a burst
        at its end; here the burst of one launch travels under the computation of the next."""

        def __init__(self):
            self.peers = [peer, parallel.PeerGather(B, 6, device, n_buffers=2)]
            self.compute = [None, torch.cuda.Stream(device)]
            self.sides = [torch.cuda.Stream(device), torch.cuda.Stream(device)]
            self.forked = False

        def __call__(self, k):
            i = k % NBUF
            cur = torch.cuda.current_stream(device)
            which = k % 2
            if which == 1 and not self.forked:
                self.compute[1].wait_stream(cur)
                self.forked = True
            stream = cur if which == 0 else self.compute[1]
            with torch.cuda.stream(stream):
                self.peers[which].solve(ik, qs[i], ts[i], ss[i], vs[i], wait=False)
                self.sides[which].wait_stream(stream)
            with torch.cuda.stream(self.sides[which]):
                self.peers[which].wait()

        def end(self):
            cur = torch.cuda.current_stream(device)
            cur.wait_stream(self.compute[1])
            for sd in self.sides:
                cur.wait_stream(sd)
            self.forked = False

        def close(self):
            self.peers[1].close()

    two = FusedTwoInFlight()
    out = {}
    for name, fn in (("serial", serial), ("overlapped", Overlapped()), ("fused", Fused()), ("fused_wait_inline", FusedSerial()),
                     ("fused_two_in_flight", two)):
        how = "graph"
        try:
            g = GraphedSteps(torch, device, fn, args.steps, end=getattr(fn, "end", None))
            run = g.run
        except Exception as exc:  # capture of the collective not possible: direct submission
            print(f"[bench] {name}: graph capture failed ({exc}); direct launches", file=sys.stderr)
            how = "direct launches"

            def run(fn=fn):
                for k in range(args.steps):
                    fn(k)
                if hasattr(fn, "end"):
                    fn.end()
        for _ in range(2):
            run()
        torch.cuda.synchronize()
        ms, _ = timed_regions(run, max(3, args.regions // 2))
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        out[name] = {"value": world * B * args.steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / args.steps,
                     "submission": how}
        g = None
    # every rank must hold every shard, bit for bit: the fused buffer against an NCCL all-gather
    step(0)
    dist.all_gather_into_tensor(gathered[0], vs[0])
    v_all, _ = peer.solve(ik, qs[0], ts[0], ss[0], vs[0])
    torch.cuda.synchronize()
    mine = gathered[0][dist.get_rank() * B:(dist.get_rank() + 1) * B]
    ok = torch.tensor([int(torch.equal(mine, vs[0])), int(torch.equal(v_all, gathered[0]))], device=device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    out["bit_equal_to_local_shard"] = bool(ok[0].item())
    out["fused_bit_equal_to_nccl_all_gather"] = bool(ok[1].item())
    out["fused_spin_timeouts"] = peer.timeouts() + two.peers[1].timeouts()
    two.close()
    peer.close()
    inbound = (world - 1) * B * 6 * 4
    out["inbound_bytes_per_rank_per_step"] = inbound
    out["nvlink_floor_us_at_900GBs"] = inbound / 900e9 * 1e6
    return out


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    from pink_b200 import FrameTask, PostureTask, _cabi, workloads
    from pink_b200.engine import get_engine
    from pink_b200.limits import ConfigurationLimit, VelocityLimit
    from pink_b200.robots import load_robot_description

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; pink_b200 has no CPU fallback")
    full_affinity = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local) if not args.no_numa_bind else "off"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    real_stdout = None
    if world > 1:
        # keep stdout to the one JSON line: NCCL prints its banner / INFO log on fd 1;
        # everything written to fd 1 from here on goes to stderr, the JSON line is written to
        # the saved descriptor at the end.  NCCL_DEBUG / NCCL_DEBUG_FILE are left as the caller set them.
        sys.stdout.flush()
        real_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=device)

    # model constants: built on rank 0, broadcast over NCCL (north_star), then
    # turned into device tables by every rank
    from pink_b200 import parallel

    robot = load_robot_description("ur5_description") if rank == 0 else None
    model = parallel.broadcast_model(robot.model if rank == 0 else None, device)
    eng = get_engine(model, device)
    table = eng.table
    B, NBUF = args.batch, args.nbuf
    f = table.frame_names.index("tool0")

    # seeded synthetic inputs, one set per buffer; rank r owns shard r of the job
    rng = np.random.default_rng(workloads.SEED + 1000 * rank)
    qs, ts, vs, ss = [], [], [], []
    for b in range(NBUF):
        q = workloads.sample_configurations(table, B, rng)
        qt = workloads.perturb_configurations(table, q, rng)
        q_d = torch.as_tensor(q, dtype=torch.float32, device=device)
        oMf, _ = eng.forward_kinematics(torch.as_tensor(qt, dtype=torch.float32, device=device))
        qs.append(q_d)
        ts.append(oMf[:, f].reshape(B, 12).contiguous())
        vs.append(torch.empty((B, 6), dtype=torch.float32, device=device))
        ss.append(torch.empty((B,), dtype=torch.int32, device=device))
    frame_task = FrameTask("tool0", position_cost=1.0, orientation_cost=1.0, lm_damping=1.0)
    frame_task.set_target(ts[0])
    posture_task = PostureTask(cost=1e-3)
    posture_task.set_target(workloads.ur5_posture_reference(model))
    limits = [ConfigurationLimit(model), VelocityLimit(model)]
    from pink_b200 import BatchedIK

    ik = BatchedIK(model, [frame_task, posture_task], workloads.UR5_DT, damping=workloads.UR5_DAMPING,
                   limits=limits, safety_break=True, device=device, batch_size=B)
    flush_buf = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=device)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def flush_l2():
        flush_buf.zero_()

    def step(k):
        i = k % NBUF
        ik.solve(qs[i], ts[i], vs[i], ss[i])

    def timed_regions(run, n_regions, pre_spin=True):
        """median and all times (ms) of `n_regions` regions, each bracketed by barrier +
        synchronize, L2 flushed before each"""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        out = []
        for _ in range(n_regions):
            flush_l2()
            barrier()
            if pre_spin:
                torch.cuda._sleep(300000)  # ~150 us: the host queues the whole region meanwhile
            e0.record()
            run()
            e1.record()
            barrier()
            out.append(e0.elapsed_time(e1))
        return float(np.median(out)), out

    # ---- device-resident throughput ("value") ---------------------------------
    for k in range(args.warmup):
        step(k)
    barrier()
    launches0 = _cabi.load().pk_launch_count()
    graphed = None
    try:
        graphed = GraphedSteps(torch, device, step, args.steps)
        graphed.run()  # upload / first-replay cost outside the timed regions
        barrier()
    except Exception as exc:  # pragma: no cover - graph capture is an optimisation only
        graphed = None
        print(f"[bench] CUDA graph submission unavailable, direct launches: {exc}", file=sys.stderr)

    def run_eager():
        for k in range(args.steps):
            step(k)

    with ClockSampler(local) as clocks:
        ms, region_ms = timed_regions(graphed.run if graphed is not None else run_eager, args.regions)
        last = (args.steps - 1) % NBUF  # the buffer set the last timed step wrote
        outputs = {"v": vs[last].cpu().numpy(), "status": ss[last].cpu().numpy()} if args.dump_outputs else None
        # keep the GPU under the same load a little longer so the sampler sees it
        t_end = time.time() + 0.5
        while time.time() < t_end:
            (graphed.run if graphed is not None else run_eager)()
            torch.cuda.synchronize()
    assert _cabi.load().pk_launch_count() - launches0 >= min(args.steps, GRAPH_CHUNK)
    bad = int(sum(int((s != 0).sum().item()) for s in ss[: min(NBUF, args.steps)]))

    # two independent batches in flight (informational): the same K launches alternated over two
    # graph branches, so that the tail of one launch (the few warps still in Cholesky rounds)
    # overlaps the start of the next.  Not the headline: `value` times serial launches.
    two_ms = None
    try:
        class TwoStreams:
            def __init__(self):
                self.side = torch.cuda.Stream(device)
                self.forked = False

            def __call__(self, k):
                cur = torch.cuda.current_stream(device)
                if k % 2 == 0:
                    step(k)
                else:
                    if not self.forked:
                        self.side.wait_stream(cur)
                        self.forked = True
                    with torch.cuda.stream(self.side):
                        step(k)

            def end(self):
                torch.cuda.current_stream(device).wait_stream(self.side)
                self.forked = False

        ts_fn = TwoStreams()
        g2 = GraphedSteps(torch, device, ts_fn, args.steps, end=ts_fn.end)
        g2.run()
        barrier()
        two_ms, _ = timed_regions(g2.run, max(3, args.regions // 2))
        two_ms /= args.steps
        g2 = None
    except Exception as exc:  # pragma: no cover
        print(f"[bench] two-stream variant unavailable: {exc}", file=sys.stderr)

    # direct-launch loop (host launch latency included), for reference
    n_direct = min(args.steps, 2000)
    eager_total, _ = timed_regions(lambda: [step(k) for k in range(n_direct)], 3, pre_spin=False)
    eager_ms = eager_total / n_direct

    # ---- end to end through host buffers ("e2e") ---------------------------------
    # Every step copies its inputs from pinned host memory and its results back, inside
    # the timed region (BatchedIK.solve_host -> pk_solve_ik_prepared_host).
    NS = max(1, args.e2e_sets)
    q_h = [torch.empty((B, 6), dtype=torch.float32).pin_memory() for _ in range(NS)]
    t_h = [torch.empty((B, 12), dtype=torch.float32).pin_memory() for _ in range(NS)]
    v_h = [torch.empty((B, 6), dtype=torch.float32).pin_memory() for _ in range(NS)]
    s_h = [torch.empty((B,), dtype=torch.int32).pin_memory() for _ in range(NS)]
    for i in range(NS):
        q_h[i].copy_(qs[i % NBUF].cpu())
        t_h[i].copy_(ts[i % NBUF].cpu())

    # --e2e-streams 2: consecutive calls alternate over two caller streams (one pinned buffer set
    # each), so that the library's two staging sets pipeline them - the upload of step k + 1
    # under the kernel and download of step k; all streams are joined before the stop event
    n_streams = max(1, min(args.e2e_streams, NS))
    user_streams = [torch.cuda.Stream(device) for _ in range(n_streams)] if n_streams > 1 else None

    def e2e_run():
        if user_streams is None:
            for k in range(args.steps):
                i = k % NS
                ik.solve_host(q_h[i], t_h[i], v_h[i], s_h[i])
            return
        cur = torch.cuda.current_stream(device)
        for st_ in user_streams:
            st_.wait_stream(cur)
        for k in range(args.steps):
            i = k % n_streams
            with torch.cuda.stream(user_streams[i]):
                ik.solve_host(q_h[i], t_h[i], v_h[i], s_h[i])
        for st_ in user_streams:
            cur.wait_stream(st_)

    # Warm-up of the host path.  The first tens of milliseconds of pinned-buffer DMA in a
    # process run 2-3x below the steady rate (measured, scripts/e2e_burst.py: 300-500 us per
    # step, then - after one driver-side stall of ~70 ms - 160 us for the rest of the process,
    # whatever the idle gaps), so W calls are not enough at the driver's W = 5: warm up in
    # batches of 20 calls for at least 0.4 s and until three consecutive batches agree within
    # 5 % of the best one (2 s at most).  The count is reported as e2e.warmup_calls.
    e2e_warm_calls, best_batch, recent = 0, float("inf"), []
    t_warm = time.time()
    while True:
        w0 = time.perf_counter()
        for k in range(20):
            ik.solve_host(q_h[k % NS], t_h[k % NS], v_h[k % NS], s_h[k % NS])
        torch.cuda.synchronize()
        batch = time.perf_counter() - w0
        e2e_warm_calls += 20
        best_batch = min(best_batch, batch)
        recent = (recent + [batch])[-3:]
        elapsed = time.time() - t_warm
        if elapsed > 2.0 or (elapsed > 0.4 and len(recent) == 3 and max(recent) <= 1.05 * best_batch):
            break
    # start-up probe of the library's host schedules under this submission pattern (same results
    # either way): three batches of K steps per schedule, the faster one stays
    host_probe = None
    if "PK_HOST_MODE" not in os.environ:
        host_probe = {}
        for mode in (0, 2):
            ik.set_host_schedule(mode)
            e2e_run()
            torch.cuda.synchronize()
            best = float("inf")
            for _ in range(3):
                w0 = time.perf_counter()
                e2e_run()
                torch.cuda.synchronize()
                best = min(best, (time.perf_counter() - w0) / args.steps)
            host_probe[mode] = best * 1e6
        ik.set_host_schedule(min(host_probe, key=host_probe.get))
    barrier()
    e2e_ms, e2e_region_ms = timed_regions(e2e_run, args.regions, pre_spin=False)
    step(0)
    torch.cuda.synchronize()
    e2e_ok = bool(torch.equal(v_h[0], vs[0].cpu()))

    # ---- solve + gather variant (multi-GPU only): v gathered on every rank --------
    gather = None
    if world > 1:
        try:
            gather = gather_variants(torch, dist, device, world, B, NBUF, step, vs, args, timed_regions, ik, qs, ts, ss)
        except Exception as exc:  # the headline line must survive a failure of the optional leg
            gather = {"error": f"{type(exc).__name__}: {exc}"}
            print(f"[bench] solve + gather variants failed: {exc}", file=sys.stderr)

    # ---- max over ranks -----------------------------------------------------------
    times = torch.tensor([ms, e2e_ms, eager_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, e2e_ms, eager_ms = (float(x) for x in times.cpu())

    if rank == 0:
        peak, peak_kind = load_peaks()
        total_steps = world * B * args.steps
        value = total_steps / (ms * 1e-3)
        kern_ms = ms / args.steps
        achieved = B * BYTES_PER_STEP / (kern_ms * 1e-3) / 1e9
        traffic, traffic_src = committed_traffic()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": kern_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args),
            "gpu_launches": int(args.steps) * world,
            "clocks": clocks.summary(),
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_kind": peak_kind,
                "kernel": ik.kernel_name() if hasattr(ik, "kernel_name") else "pk::ik_chain_kernel<6,1>",
                "kernel_ms": kern_ms,
                "timing": (f"{graphed.describe()} per timed region" if graphed is not None else "direct launches")
                          + f"; median of {args.regions} regions of {args.steps} steps, L2 flushed before each",
                "region_ms": region_ms,
                "eager_ms_per_step": eager_ms,
                "two_batches_in_flight_ms_per_step": two_ms,
                "algorithmic_bytes_per_launch": B * BYTES_PER_STEP,
                "l2": f"{NBUF} rotating input/output sets ({NBUF * B * BYTES_PER_STEP / 2**20:.0f} MiB) and a "
                      f"{2 * L2_BYTES / 2**20:.0f} MiB write between regions (L2 = 126 MiB)",
            },
            "e2e": {
                "value": world * B * args.steps / (e2e_ms * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": B * (6 + 12) * 4, "d2h_bytes_per_step": B * (6 + 1) * 4,
                "ms_per_step": e2e_ms / args.steps, "region_ms": e2e_region_ms, "warmup_calls": e2e_warm_calls,
                "bitwise_equal_to_device_path": e2e_ok,
                "api": "BatchedIK.solve_host -> pk_solve_ik_prepared_host (pinned host buffers, %d set(s), %d caller stream(s); schedule %s)"
                       % (NS, n_streams, getattr(ik, "host_schedule", os.environ.get("PK_HOST_MODE", "0"))),
                "schedule_probe_us_per_call": host_probe,
                "numa": numa,
            },
            "nonzero_status": bad,
        }
        if gather is not None:
            line["solve_plus_allgather"] = gather
            for g in gather.values():
                if isinstance(g, dict) and "value" in g:
                    g["efficiency_vs_solve_only"] = g["value"] / value
        if not args.no_configs and world == 1:
            try:
                line["configs"] = humanoid_configs(torch, device, peak)
            except Exception as exc:  # the headline line must survive a failure here
                line["configs"] = {"error": f"{type(exc).__name__}: {exc}"}
        if not args.no_cpu and world == 1:
            os.sched_setaffinity(0, full_affinity)  # the CPU arm gets every core again
            line["cpu_baseline"] = cpu_baseline_block(B)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        if real_stdout is not None:
            os.write(real_stdout, (json.dumps(line) + "\n").encode())
        else:
            print(json.dumps(line), flush=True)
    # release the captured graphs and the prepared problem before the process group goes
    graphed = None
    ik = None
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--nbuf", type=int, default=32)
    ap.add_argument("--regions", type=int, default=7, help="timed regions of K steps each; the median is reported")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the humanoid configs block (N = 1 only)")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--e2e-sets", type=int, default=2, help="pinned host buffer sets the e2e steps rotate over")
    ap.add_argument("--e2e-streams", type=int, default=2, help="caller streams the e2e steps alternate over (2: consecutive calls pipeline through the library's two staging sets)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write v and status of the last one (rank 0's shard) as DIR/<name>.npy; "
                         "--impl ours dumps input set (steps - 1) %% nbuf, --impl reference its one workload, so the two "
                         "dump the same instances only when steps %% nbuf == 1")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()

"""Parity THROUGH THE KERNELS bench.py TIMES: the persistent TMA-staged stepping kernel
(`uav_step_staged_kernel`, csrc/step_kernel.cuh) is only chosen for batches with more tiles than the
persistent grid (> 56,832 UAVs at 3 CTAs/SM, > 37,888 at 2), a uniform input mode and one parameter set.
Every test here asserts — through mrsb_get_step_info — that the staged kernel really ran, then
compares it with

  * the CPU oracle (UavSystem::makeStep, uav_system.hpp:304-380 + multirotor_model.hpp:220-286) at
    BASELINE sizes within helpers.TOL after 10 s of simulated flight, and
  * the direct kernel (`MRSB_NO_STAGING=1`, read per launch) BIT FOR BIT, including a partial last
    tile, UAVs with the one-way take-off patch flag (MM:264-277) and UAVs whose v_prev differs from v
    (after setState, MM:424-433).
"""
import os

import numpy as np
import pytest

from helpers import TOL, assert_parity, make_pair, rand
from oracle import binding as O

pytestmark = pytest.mark.gpu

THREADS = os.cpu_count() or 1
FIELDS = ("x", "v", "R", "omega", "motor_rpm", "v_prev", "imu")


def af(name, **kw):
    from mrs_multirotor_simulator_b200 import airframe

    return airframe(name, **kw)


def big_grid(n, z, pitch=4.0):
    side = int(np.ceil(np.sqrt(n)))
    i = np.arange(n)
    return np.stack([pitch * (i % side), pitch * (i // side), np.full(n, z)], axis=1).astype(np.float64)


def commands(mode, n, seed=42):
    r = lambda s, lo, hi: rand(seed, s, n, lo, hi)
    if mode == O.ACTUATOR_CMD:
        return np.stack([rand(seed, 10 + m, n, 0.4, 0.7) for m in range(8)], axis=1)
    if mode == O.VELOCITY_HDG_RATE_CMD:
        return np.stack([r(1, -2, 2), r(2, -2, 2), r(3, 0, 2), r(4, -1, 1)], axis=1)
    if mode == O.VELOCITY_HDG_CMD:
        return np.stack([r(1, -2, 2), r(2, -2, 2), r(3, -2, 2), r(4, -np.pi, np.pi)], axis=1)
    if mode == O.POSITION_CMD:
        return np.stack([r(1, -10, 10), r(2, -10, 10), r(3, 2, 12), r(4, -3.1, 3.1)], axis=1)
    raise ValueError(mode)


def assert_staged(gpu, mode, nm):
    info = gpu.step_info()
    assert info["variant"] == "staged" and info["mode"] == mode and info["n_motors"] == nm, info


def test_c3_at_its_real_size_velocity_hdg_k10():
    """BASELINE config 3 as written: 65,536 x500 on a 256 x 256 grid at z = 10, random VelocityHdgCmd, collisions and
    ground off, dt = 0.01, K = 10 fused substeps per launch, 100 launches = 10 s — staged kernel <4, VELOCITY_HDG, K>1>."""
    n = 65536
    orc, gpu = make_pair([af("x500")], None, big_grid(n, 10.0))
    cmd = commands(O.VELOCITY_HDG_CMD, n)
    orc.set_input(O.VELOCITY_HDG_CMD, cmd)
    gpu.set_input(O.VELOCITY_HDG_CMD, cmd)
    orc.make_step(0.01, 1000, n_threads=THREADS)
    for _ in range(100):
        gpu.make_step(0.01, 10)
    assert_staged(gpu, O.VELOCITY_HDG_CMD, 4)
    assert_parity(orc, gpu, what="C3 at 65,536 UAVs")


def test_c4_headline_instantiation_velocity_hdg_rate_k1_10s():
    """The kernel behind BENCH's `value`: <4, VELOCITY_HDG_RATE, K=1> staged, on a slab of the C4 swarm (x500, ground
    plane at z = 0, the two zero-actuator warm-up steps of uav_system_ros.cpp:223-232, bench.py's command distribution),
    131,072 + 57 UAVs (partial last tile), 1000 ticks = 10 s."""
    n = 131072 + 57
    x500 = af("x500", ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=False, g=9.81)
    orc, gpu = make_pair([x500], None, big_grid(n, 0.0))
    cmd = commands(O.VELOCITY_HDG_RATE_CMD, n)
    for s in (orc, gpu):
        s.set_input(O.ACTUATOR_CMD, np.zeros((n, 8)))
    orc.make_step(0.01, 2, n_threads=THREADS)
    gpu.make_step(0.01)
    gpu.make_step(0.01)
    orc.set_input(O.VELOCITY_HDG_RATE_CMD, cmd)
    gpu.set_input(O.VELOCITY_HDG_RATE_CMD, cmd)
    orc.make_step(0.01, 1000, n_threads=THREADS)
    for _ in range(1000):
        gpu.make_step(0.01)
    assert_staged(gpu, O.VELOCITY_HDG_RATE_CMD, 4)
    assert_parity(orc, gpu, what="C4 headline kernel at 131,129 UAVs")


@pytest.mark.parametrize("frame,nm", [("x500", 4), ("f550", 6), ("naki", 8)])
def test_c5_actuator_cmd_staged_10s(frame, nm):
    """BASELINE config 5's kernels, one airframe at a time (the uniform staged instantiations <4|6|8, ACTUATOR, K=1>):
    open-loop motors ~U(0.4, 0.7) re-drawn every 100 steps, ground on, 58,001 UAVs, 10 s.  Open-loop flight is unstable
    (tumbling, km-scale drift), so x and v are compared relative to the excursion like tests/test_step_parity.py."""
    n = 58001
    orc, gpu = make_pair([af(frame, ground_enabled=True)], None, big_grid(n, 0.0))
    for block in range(10):
        cmd = commands(O.ACTUATOR_CMD, n, seed=100 + block)
        orc.set_input(O.ACTUATOR_CMD, cmd)
        gpu.set_input(O.ACTUATOR_CMD, cmd)
        orc.make_step(0.01, 100, n_threads=THREADS)
        for _ in range(100):
            gpu.make_step(0.01)
    assert_staged(gpu, O.ACTUATOR_CMD, nm)
    so, sg = orc.get_state(), gpu.get_full_state()
    for k in ("x", "v", "omega"):
        scale = 1.0 + np.max(np.abs(so[k]))
        assert np.max(np.abs(so[k] - sg[k])) <= 1e-7 * scale, k
    assert np.max(np.abs(so["motor_rpm"] - sg["motor_rpm"])) <= 1e-5


def test_position_cmd_staged_10s():
    """<4, POSITION, K=1> staged (2 CTAs/SM: every PID row is live) on 58,001 x500s flying to seeded waypoints, 10 s."""
    n = 58001
    orc, gpu = make_pair([af("x500")], None, big_grid(n, 5.0), rand(3, 0, n, -3, 3))
    cmd = commands(O.POSITION_CMD, n)
    cmd[:, :2] += big_grid(n, 0.0)[:, :2]
    orc.set_input(O.POSITION_CMD, cmd)
    gpu.set_input(O.POSITION_CMD, cmd)
    orc.make_step(0.01, 1000, n_threads=THREADS)
    for _ in range(1000):
        gpu.make_step(0.01)
    assert_staged(gpu, O.POSITION_CMD, 4)
    assert_parity(orc, gpu, what="PositionCmd staged")


FF_KIND = {"acceleration_hdg_rate": 0, "acceleration_hdg": 1, "velocity_hdg": 2, "velocity_hdg_rate": 3}  # the oracle's numbering
DT_PHASES = (0.01, 0.005, 0.02)  # the edited flights change dt twice: DevParams::filt of the set passed by value must follow


def edited_airframe(frame):
    """The airframe with every constant the kernel derives something from changed: mass, kf, km, tau, drag, ground_z, and a
    symmetric positive-definite J with off-diagonal terms (the j_diagonal == 0 branch of derivative(), step_kernel.cuh)."""
    d = af(frame, ground_enabled=True, ground_z=-0.25, takeoff_patch_enabled=True)
    d.update(mass=1.13 * d["mass"], kf=1.07 * d["kf"], km=0.9 * d["km"], motor_time_constant=0.04, air_resistance_coeff=0.35)
    m, a, bh = d["mass"], d["arm_length"], d["body_height"]
    jxy, jz = m * (3.0 * a * a + bh * bh) / 12.0, m * a * a / 2.0
    J = np.array([[jxy, 0.12 * jxy, -0.08 * jxy], [0.12 * jxy, 1.1 * jxy, 0.1 * jxy], [-0.08 * jxy, 0.1 * jxy, jz]])
    assert np.all(np.linalg.eigvalsh(J) > 0)
    d["J"] = J.tolist()
    return d


def apply_edits(s, gidx, frame, edits):
    """Batch-wide edits of the "edited" flights on a system that holds the UAVs `gidx` of the batch (all of them, or the oracle's
    sample): set_params with edited_airframe, then all five gain sets with every ki != 0 (rate included: the three rate-integral rows
    become live), an external moment on a third of the UAVs and the four feed-forwards on overlapping subsets (UAVs with both
    acceleration feed-forwards take each branch of use_a / use_ar, step_kernel.cuh).  edits == "no_desaturation": the mixer's
    desaturation off as well."""
    gpu = not isinstance(s, O.OracleSwarm)
    sel = lambda mask: np.flatnonzero(mask).astype(np.int32)
    u = lambda stream, idx, lo, hi: lo + (hi - lo) * O.u01(31, stream, gidx[idx])
    s.set_params(edited_airframe(frame))
    s.set_controller_params("rate", [4.2, 0.045, 0.6])
    s.set_controller_params("attitude", [6.5, 0.06, 0.05, 9.0, 1.2])
    s.set_controller_params("velocity", [2.2, 0.06, 0.05, 4.5])
    s.set_controller_params("position", [1.8, 0.12, 0.25, 5.0])
    if edits == "no_desaturation":
        s.set_controller_params("mixer", [0.0])
    m = sel(gidx % 3 == 2)
    s.set_external_moment(np.stack([u(0, m, -0.02, 0.02), u(1, m, -0.02, 0.02), u(2, m, -0.01, 0.01)], axis=1), idx=m)
    for stream, (kind, mask) in enumerate([("acceleration_hdg", gidx % 4 < 2), ("acceleration_hdg_rate", (gidx % 4 == 1) | (gidx % 4 == 2)),
                                           ("velocity_hdg", gidx % 5 < 2), ("velocity_hdg_rate", (gidx % 5 == 1) | (gidx % 5 == 2))]):
        i = sel(mask)
        ff = np.stack([u(10 + 4 * stream + c, i, -0.3, 0.3) for c in range(4)], axis=1)
        s.set_feedforward(kind if gpu else FF_KIND[kind], ff, idx=i)


def setup_flight(s, gidx, n, frame, mode, edits):
    """The flight's set-up on a system that holds the UAVs `gidx` of an n-UAV batch: every UAV on the ground with the take-off patch
    flag; a third given a state whose v_prev differs from v (FLAG_VPREV) and a tilted, spinning start in the air; the command of
    `mode`; a few crashed UAVs; an external force on everybody; then the edits, if any."""
    sel = lambda mask: np.flatnonzero(mask).astype(np.int32)
    idx = sel(gidx % 3 == 0)
    k3 = gidx[idx] // 3  # position in arange(0, n, 3)
    u = lambda stream, lo, hi: lo + (hi - lo) * O.u01(5, stream, k3)
    st = s.get_state(idx)
    x = st["x"] + np.stack([np.zeros(len(idx)), np.zeros(len(idx)), u(1, 0.5, 6.0)], axis=1)
    v = np.stack([u(2, -2, 2), u(3, -2, 2), u(4, -1, 1)], axis=1)
    w = np.stack([u(5, -0.5, 0.5), u(6, -0.5, 0.5), u(7, -0.5, 0.5)], axis=1)
    s.set_state(idx, x=x, v=v, omega=w)
    s.set_input(mode, commands(mode, n)[gidx])
    s.crash(sel(gidx % 997 == 5))  # 5, 1002, 1999, ...
    s.apply_force(np.stack([rand(5, 8, n, -1, 1), rand(5, 9, n, -1, 1), rand(5, 10, n, -1, 1)], axis=1)[gidx])
    if edits:
        apply_edits(s, gidx, frame, edits)


def flight_phases(launches, edits):
    """(dt, launches) of a flight: dt = 0.01 throughout, or the edited flights' three dt phases."""
    if not edits:
        return [(0.01, launches)]
    split = [launches - 2 * (launches // 3), launches // 3, launches // 3]
    return list(zip(DT_PHASES, split))


def spawn_of(n):
    return big_grid(n, 0.0), rand(5, 0, n, -3, 3)


def _run_variant(staging, frame, mode, k, n, launches, edits=None):
    """One flight on the GPU with or without the staged kernel; returns (full state, crash flags, the variant that ran in each dt
    phase)."""
    from mrs_multirotor_simulator_b200 import UavBatch

    if staging:
        os.environ.pop("MRSB_NO_STAGING", None)
    else:
        os.environ["MRSB_NO_STAGING"] = "1"
    try:
        a = af(frame, ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=True)  # FLAG_TAKEOFF on every UAV at spawn
        xyz, hdg = spawn_of(n)
        b = UavBatch([a], spawn_xyz=xyz, spawn_heading=hdg, n=n)
        setup_flight(b, np.arange(n), n, frame, mode, edits)
        infos = []
        for dt, count in flight_phases(launches, edits):
            for _ in range(count):
                b.make_step(dt, k)
            infos.append(b.step_info())
        out = b.get_full_state()
        out["crashed"] = b.has_crashed()
        takeoff = np.array([b.get_params(int(i)).takeoff_patch_enabled for i in (0, 1, 2, 3, n - 1)])
        out["takeoff_flag_sample"] = takeoff
        b.close()
        return out, infos
    finally:
        os.environ.pop("MRSB_NO_STAGING", None)


@pytest.mark.parametrize("edits", [None, "edited", "no_desaturation"])
@pytest.mark.parametrize("frame,nm", [("x500", 4), ("f550", 6), ("naki", 8)])
@pytest.mark.parametrize("mode", [O.ACTUATOR_CMD, O.VELOCITY_HDG_RATE_CMD, O.VELOCITY_HDG_CMD, O.POSITION_CMD])
@pytest.mark.parametrize("k", [1, 10])
def test_staged_equals_direct_bit_for_bit(frame, nm, mode, k, edits):
    """Same swarm, same calls, staged kernel vs MRSB_NO_STAGING=1 (direct kernel): every state component, IMU, v_prev
    and crash flag identical in every bit.  58,001 UAVs: 454 tiles, the last one holds 17 UAVs.  `edits`: the flights of
    apply_edits (the staged kernel's parameter set passed by value after set_params and gain edits, live rate integrals, external
    moments, feed-forwards), flown at dt = 0.01, 0.005, 0.02 in turn; the staged kernel must run in every dt phase."""
    n = 58001
    launches = 40 if k == 1 else 6
    direct, info_d = _run_variant(False, frame, mode, k, n, launches, edits)
    staged, info_s = _run_variant(True, frame, mode, k, n, launches, edits)
    for d, s in zip(info_d, info_s):
        assert d["variant"] == "direct", d
        assert s["variant"] == "staged" and s["n_motors"] == nm and s["mode"] == mode, s
    for key in direct:
        assert np.array_equal(direct[key], staged[key], equal_nan=True), f"{key} differs between the staged and the direct kernel"
    assert np.all(np.isfinite(staged["x"]))


def test_c5_interleaved_airframes_run_the_staged_kernels_per_bucket():
    """BASELINE config 5 as written: x500 / f550 / naki INTERLEAVED by index, ActuatorCmd re-drawn every 100 steps, ground on.
    The library buckets the batch by airframe at create, so every airframe's UAVs run their uniform staged kernel
    (<4|6|8, ACTUATOR, K=1>; 3 x 58,001 UAVs) — against the oracle (which knows nothing of buckets), 5 s."""
    n = 3 * 58001
    types = [af("x500", ground_enabled=True), af("f550", ground_enabled=True), af("naki", ground_enabled=True)]
    tou = (np.arange(n) % 3).astype(np.int32)
    orc, gpu = make_pair(types, tou, big_grid(n, 0.0))
    for block in range(5):
        cmd = commands(O.ACTUATOR_CMD, n, seed=200 + block)
        orc.set_input(O.ACTUATOR_CMD, cmd)
        gpu.set_input(O.ACTUATOR_CMD, cmd)
        orc.make_step(0.01, 100, n_threads=THREADS)
        for _ in range(100):
            gpu.make_step(0.01)
    info = gpu.step_info()
    assert info["variant"] == "staged" and info["mode"] == O.ACTUATOR_CMD and info["n_motors"] == 8, info  # the last bucket launched: naki
    so, sg = orc.get_state(), gpu.get_full_state()
    for k in ("x", "v", "omega"):
        scale = 1.0 + np.max(np.abs(so[k]))
        assert np.max(np.abs(so[k] - sg[k])) <= 1e-7 * scale, k
    assert np.max(np.abs(so["motor_rpm"] - sg["motor_rpm"])) <= 1e-5

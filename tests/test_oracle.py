"""CPU-only checks of the oracle (oracle/): golden fixtures, the reference-generated collision
fixture, the real vendored nanoflann vs the cell-list port, and analytic known-answer tests derived
from the reference source (SURVEY §4 item 2, App. A.9 quirk list)."""
import json
import os

import numpy as np
import pytest

from helpers import digest, rand
from mrs_multirotor_simulator_b200.airframes import AIRFRAMES, airframe
from oracle import binding as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    with open(os.path.join(GOLD, name)) as f:
        return json.load(f)


def one(frame="x500", pos=(0, 0, 5), hdg=0.0, **kw):
    return O.OracleSwarm([airframe(frame, **kw)], spawn_xyz=[list(pos)], spawn_heading=[hdg], n=1)


# ---------------------------------------------------------------- golden fixtures
# The trajectory fixtures are the output of the reference's own UavSystem sources (make_golden.py), which the restatement
# follows bit for bit: the comparison is exact.
def test_golden_c1_trajectory():
    g = load("c1_position_x500.json")
    s = one("x500", g["spawn"], g["heading"])
    s.set_input(O.POSITION_CMD, [g["cmd"]])
    for smp in g["samples"]:
        s.make_step(g["dt"], 200)
        st = s.get_state()
        for k in ("x", "v", "R", "omega", "motor_rpm", "imu"):
            assert np.array_equal(st[k][0], np.array(smp[k])), (smp["t"], k)
    # independent numpy restatement made during the survey (SURVEY App. D)
    assert np.allclose(st["x"][0], [4.99966878, -2.99316222, 3.99492282], atol=1e-8)


def test_golden_every_mode_every_motor_count():
    g = load("modes_2s.json")
    assert len(g["cases"]) == 30
    for c in g["cases"]:
        s = one(c["frame"], g["spawn"], g["heading"])
        s.set_input(c["mode_id"], [c["cmd"]])
        s.make_step(c["dt"], c["steps"])
        st = s.get_state()
        for k in ("x", "v", "R", "omega", "motor_rpm", "imu"):
            assert np.array_equal(st[k][0], np.array(c[k])), (c["frame"], c["mode"], k)


def test_reference_generated_collision_fixture_vs_port():
    """tests/golden/collisions_400.json was produced by the reference's real nanoflann."""
    g = load("collisions_400.json")
    xyz = np.array(g["xyz"])
    tou = np.array(g["type_of_uav"])
    arm = np.array([airframe(f)["arm_length"] for f in g["frames"]])[tou]
    prop = np.array([airframe(f)["prop_radius"] for f in g["frames"]])[tou]
    mass = np.array([airframe(f)["mass"] for f in g["frames"]])[tou]
    pairs, forces, _ = O.collide_snapshot(xyz, arm, prop, mass, False, g["rebounce"], engine="port")
    _, _, crashed = O.collide_snapshot(xyz, arm, prop, mass, True, g["rebounce"], engine="port")
    pairs = pairs[np.lexsort((pairs[:, 1], pairs[:, 0]))]
    assert pairs.tolist() == g["pairs"] and len(pairs) > 50
    assert crashed.astype(int).tolist() == g["crashed"]
    assert np.allclose(forces, np.array(g["forces"]), rtol=1e-12, atol=0)


@pytest.mark.parametrize("n,scale", [(1, 1.0), (2, 0.01), (400, 0.5), (5000, 0.3), (40000, 0.35)])
def test_port_equals_real_nanoflann(n, scale):
    """Against the reference's nanoflann where oracle/_ref/libref_nanoflann.so is built; otherwise against the stored digests
    of the results that comparison accepted (golden/nanoflann_port_digests.json: pairs and crash flags equal to nanoflann's,
    forces within 1e-11 of them)."""
    side = int(np.ceil(np.sqrt(n)))
    k = np.arange(n)
    xyz = np.stack([scale * (4.0 * (k % side) + rand(3, 0, n, -2, 2)), scale * (4.0 * (k // side) + rand(3, 1, n, -2, 2)), rand(3, 2, n, 2, 4)], axis=1)
    frames = list(AIRFRAMES)
    tou = (k * 7) % len(frames)
    arm = np.array([AIRFRAMES[f]["arm_length"] for f in frames])[tou]
    prop = np.array([AIRFRAMES[f]["prop_radius"] for f in frames])[tou]
    mass = np.array([AIRFRAMES[f]["mass"] for f in frames])[tou]
    for crash in (False, True):
        b = O.collide_snapshot(xyz, arm, prop, mass, crash, 100.0, engine="port", n_threads=4)
        pb = b[0][np.lexsort((b[0][:, 1], b[0][:, 0]))] if len(b[0]) else b[0]
        if O.ref_lib() is None:
            stored = load("nanoflann_port_digests.json")["cases"][f"{n}-{scale}-{int(crash)}"]
            assert [digest(pb), digest(b[2]), digest(b[1])] == stored, "pairs, crash flags, forces"
            continue
        a = O.collide_snapshot(xyz, arm, prop, mass, crash, 100.0, engine="nanoflann", n_threads=4)
        pa = a[0][np.lexsort((a[0][:, 1], a[0][:, 0]))] if len(a[0]) else a[0]
        assert np.array_equal(pa, pb)
        assert np.array_equal(a[2], b[2])
        assert np.allclose(a[1], b[1], rtol=1e-11, atol=0)


# ---------------------------------------------------------------- analytic known answers
def test_spawn_rotation_is_rz_of_minus_heading():
    """multirotor_model.hpp:439-446: R = AngleAxis(-heading, z)  =>  R(0,1) = sin h, R(1,0) = -sin h."""
    h = 0.7
    R = one(hdg=h).get_state()["R"][0].reshape(3, 3).T
    assert np.allclose(R, [[np.cos(h), np.sin(h), 0], [-np.sin(h), np.cos(h), 0], [0, 0, 1]], atol=1e-15)


def test_motor_lag_is_discrete_first_order_outside_the_ode():
    """multirotor_model.hpp:244-246: rpm' = a rpm + (1-a) u, a = exp(-dt/tau); idle is rpm_min (:408)."""
    s = one()
    p = airframe("x500")
    cmd = np.array([[0.2, 0.4, 0.6, 0.8, 0, 0, 0, 0]])
    s.set_input(O.ACTUATOR_CMD, cmd)
    a = np.exp(-0.01 / p["motor_time_constant"])
    rpm = np.zeros(4)
    for _ in range(5):
        s.make_step(0.01)
        u = p["min_rpm"] + (p["max_rpm"] - p["min_rpm"]) * cmd[0, :4]
        rpm = a * rpm + (1 - a) * u
        assert np.allclose(s.get_state()["motor_rpm"][0, :4], rpm, rtol=1e-14)
    s.set_input(O.INPUT_UNKNOWN)
    s.make_step(0.01, 400)
    assert np.allclose(s.get_state()["motor_rpm"][0, :4], p["min_rpm"], rtol=1e-6)


@pytest.mark.parametrize("frame", ["x500", "f550", "naki"])
def test_hover_equilibrium(frame):
    """thrust row = kf * sum(rpm^2)  =>  at rpm_h = sqrt(m g / (n kf)) the UAV neither climbs nor sinks."""
    p = airframe(frame)
    n = p["n_motors"]
    rpm_h = np.sqrt(p["mass"] * 9.81 / (n * p["kf"]))
    u = (rpm_h - p["min_rpm"]) / (p["max_rpm"] - p["min_rpm"])
    s = one(frame)
    rpm = np.zeros((1, 8))
    rpm[0, :n] = rpm_h
    s.set_state(motor_rpm=rpm)
    s.set_input(O.ACTUATOR_CMD, np.full((1, 8), u))
    s.make_step(0.01, 200)
    st = s.get_state()
    assert np.max(np.abs(st["v"])) < 1e-9 and np.max(np.abs(st["x"][0] - [0, 0, 5])) < 1e-9
    assert np.allclose(st["imu"][0], [0, 0, 9.81], atol=1e-8)


def test_mixer_matrix_x500():
    m = one().get_mixer_allocation()[:4]
    r = np.sqrt(0.5)
    assert np.allclose(m, [[-r, -r, -1, 1], [r, r, -1, 1], [r, -r, 1, 1], [-r, r, 1, 1]], atol=1e-12)


def test_pid_truth_table():
    """pid.hpp:67-96: derivative kick, inclusive saturation, integrate AFTER the output and only if |u| < antiwindup."""
    st = np.zeros(2)
    u = O.pid_update(st, 2.0, 0.5, 0.1, 60.0, 1.0, 0.2, 0.01)  # first call: last_error = 0 -> derivative kick
    assert u == 2.0 * 0.2 + 0.5 * (0.2 / 0.01) + 0.1 * 0.0
    assert st[0] == 0.2 and st[1] == 0.0  # |u| = 10.4 >= antiwindup: no integration
    st = np.array([0.2, 0.0])
    u = O.pid_update(st, 2.0, 0.5, 0.1, 6.0, 1.0, 0.2, 0.01)
    assert u == 0.4 and st[1] == 0.2 * 0.01  # |u| < 1: integrate after computing u
    st = np.array([3.0, 0.0])
    assert O.pid_update(st, 2.0, 0.0, 0.0, 6.0, 1.0, 3.0, 0.01) == 6.0  # u == sat exactly -> clamps (>=)
    st = np.array([-4.0, 0.0])
    assert O.pid_update(st, 2.0, 0.0, 0.0, 6.0, 1.0, -4.0, 0.01) == -6.0
    st = np.array([50.0, 0.0])
    assert O.pid_update(st, 2.0, 0.0, 0.0, -1.0, 1.0, 50.0, 0.01) == 100.0  # saturation <= 0: unlimited (rate controller)
    st = np.array([0.1, 0.5])
    O.pid_update(st, 1.0, 0.0, 0.0, 6.0, -1.0, 0.1, 0.01)
    assert st[1] == 0.5  # antiwindup <= 0: the integral never moves


def test_ground_clamp_and_takeoff_patch_is_one_way():
    s = one("x500", (0, 0, 0.0), ground_enabled=True, ground_z=0.0)
    s.make_step(0.01, 100)
    st = s.get_state()
    assert st["x"][0, 2] == 0.0 and not st["v"].any() and not st["omega"].any()
    s = one("x500", (0, 0, 3.0), takeoff_patch_enabled=True)
    s.make_step(0.01, 50)
    assert s.get_state()["x"][0, 2] == 3.0 and s.get_params(0).takeoff_patch_enabled == 1
    s.set_input(O.VELOCITY_HDG_RATE_CMD, [[0, 0, 1.0, 0]])
    s.make_step(0.01, 300)
    assert s.get_params(0).takeoff_patch_enabled == 0 and s.get_state()["x"][0, 2] > 4.0
    s.set_input(O.INPUT_UNKNOWN)
    s.make_step(0.01, 300)
    assert s.get_state()["x"][0, 2] < 0.0  # the platform is gone for good (multirotor_model.hpp:275)


def test_negative_thrust_request_gives_nan_throttle_then_idle_motors():
    """acceleration_controller.hpp:117-120: sqrt of a negative thrust -> NaN -> zeroed by MM:398-400."""
    s = one()
    s.set_input(O.ACCELERATION_HDG_RATE_CMD, [[0, 0, -30.0, 0]])
    s.make_step(0.01, 300)
    st = s.get_state()
    assert np.all(np.isfinite(st["x"])) and np.allclose(st["motor_rpm"][0, :4], 1170.0, rtol=1e-3)


def test_attitude_error_vector():
    """attitude_controller.hpp:82-89: E = 1/2 (Rd^T R - R^T Rd), e = ((E12-E21)/2, ...)  =>  from level, a desired roll th gives e_x = sin(th)."""
    th = 0.2
    Rd = np.array([[1, 0, 0], [0, np.cos(th), -np.sin(th)], [0, np.sin(th), np.cos(th)]])
    s = one()
    s.set_input(O.ATTITUDE_CMD, [list(Rd.T.reshape(9)) + [0.5]])
    s.make_step(0.01)
    pid = s.get_pid_state(0)
    assert np.isclose(pid[12], np.sin(th), atol=1e-15)  # attitude x last_error
    assert pid[14] == 0.0 and pid[16] == 0.0


def test_rk4_is_fourth_order():
    """Torque-free spinning body under constant thrust: halving dt divides the error by ~16."""
    def run(dt):
        s = one()
        rpm = np.zeros((1, 8))
        rpm[0, :4] = 4000.0
        u = (4000.0 - 1170.0) / (7800.0 - 1170.0)
        s.set_state(motor_rpm=rpm, omega=[[0.9, -1.3, 2.1]], v=[[1.0, 2.0, -0.5]])
        s.set_input(O.ACTUATOR_CMD, np.full((1, 8), u))
        s.make_step(dt, int(round(0.8 / dt)))
        st = s.get_state()
        return np.concatenate([st["x"][0], st["R"][0]])
    ref = run(0.0005)
    e1, e2 = np.max(np.abs(run(0.02) - ref)), np.max(np.abs(run(0.01) - ref))
    assert 11.0 < e1 / e2 < 22.0, e1 / e2


def test_set_params_resets_gains_and_pid_state():
    s = one()
    s.set_controller_params("position", [1.0, 0.0, 0.5, 3.0])
    s.set_input(O.POSITION_CMD, [[1, 1, 6, 0]])
    s.make_step(0.01, 50)
    assert s.get_pid_state(0)[1] != 0.0
    s.set_params(airframe("x500", mass=2.2))  # uav_system.hpp:404-409
    assert not s.get_pid_state(0).any()
    a = one()
    a.set_params(airframe("x500", mass=2.2))
    for sw in (s, a):
        sw.set_input(O.POSITION_CMD, [[1, 1, 6, 0]])
    st0 = s.get_state()
    a.set_state(x=st0["x"], v=st0["v"], R=st0["R"], omega=st0["omega"], motor_rpm=st0["motor_rpm"])
    s.make_step(0.01, 20)
    a.make_step(0.01, 20)
    # same gains (defaults) and same PID state from here on; v_prev differs (setState leaves it), so compare x
    assert np.allclose(s.get_state()["x"], a.get_state()["x"], atol=1e-12)


def test_coincident_uavs_collide_with_zero_force_and_self_is_skipped():
    xyz = np.array([[1.0, 1.0, 1.0], [1.0, 1.0, 1.0], [9.0, 9.0, 9.0]])
    pairs, forces, crashed = O.collide_snapshot(xyz, 0.25, 0.15, 2.0, False, 100.0, engine="port")
    assert sorted(map(tuple, pairs)) == [(0, 1), (1, 0)] and not forces.any()
    _, _, crashed = O.collide_snapshot(xyz, 0.25, 0.15, 2.0, True, 100.0, engine="port")
    assert crashed.tolist() == [1, 1, 0]


def test_squared_distance_is_compared_with_unsquared_lengths():
    """multirotor_simulator.cpp:326,346: radius 3.0 and crit (= 0.8 m for two x500) are compared with d^2."""
    for d, hit in ((0.89, True), (0.90, False), (1.5, False)):  # sqrt(0.8) = 0.8944
        xyz = np.array([[0.0, 0.0, 2.0], [d, 0.0, 2.0]])
        pairs, _, _ = O.collide_snapshot(xyz, 0.25, 0.15, 2.0, False, 100.0, engine="port")
        assert (len(pairs) == 2) == hit, d


# ---------------------------------------------------------------- ROS-wrapper rows (uav_system_ros.cpp)
def test_odometry_quaternion_and_body_frame_velocity():
    s = one(hdg=0.0)
    yaw = 0.6
    R = np.array([[np.cos(yaw), -np.sin(yaw), 0], [np.sin(yaw), np.cos(yaw), 0], [0, 0, 1]])
    s.set_state(R=[R.T.reshape(9)], v=[[1.0, 2.0, 3.0]], omega=[[0.1, 0.2, 0.3]])
    od = s.get_odometry()[0]
    assert np.allclose(od[:3], [0, 0, 5])
    assert np.allclose(od[3:7], [0, 0, np.sin(yaw / 2), np.cos(yaw / 2)], atol=1e-15)  # x y z w
    assert np.allclose(od[7:10], R.T @ [1.0, 2.0, 3.0], atol=1e-15) and np.allclose(od[10:13], [0.1, 0.2, 0.3])
    for Rm, q in (([[1, 0, 0], [0, -1, 0], [0, 0, -1]], [1, 0, 0, 0]), ([[-1, 0, 0], [0, 1, 0], [0, 0, -1]], [0, 1, 0, 0]),
                  ([[-1, 0, 0], [0, -1, 0], [0, 0, 1]], [0, 0, 1, 0])):  # the three trace <= 0 branches
        s.set_state(R=[np.array(Rm, dtype=float).T.reshape(9)])
        assert np.allclose(s.get_odometry()[0, 3:7], q, atol=1e-15)


def test_rangefinder_model():
    s = one(pos=(0, 0, 5), ground_enabled=True, ground_z=1.0)
    assert np.isclose(s.get_rangefinder()[0, 0], 4.0 + 0.01, atol=1e-12)
    th = 0.4
    R = np.array([[1, 0, 0], [0, np.cos(th), -np.sin(th)], [0, np.sin(th), np.cos(th)]])
    s.set_state(R=[R.T.reshape(9)])
    assert np.isclose(s.get_rangefinder()[0, 0], 4.0 / np.cos(th) + 0.01, atol=1e-12)
    s.set_state(x=[[0, 0, 60.0]])
    assert s.get_rangefinder()[0, 0] == 41.0  # beyond 40 m
    s.set_state(x=[[0, 0, 5.0]], R=[np.diag([1.0, -1.0, -1.0]).reshape(9)])
    assert s.get_rangefinder()[0, 0] == 41.0  # inverted


def test_timeout_input_holds_position_and_heading():
    s = one(hdg=0.0)
    s.set_input(O.POSITION_CMD, [[30.0, 0.0, 5.0, 0.0]])
    s.make_step(0.01, 150)
    x0 = s.get_state()["x"][0].copy()
    assert x0[0] > 2.0
    s.timeout_input()
    s.make_step(0.01, 1500)
    st = s.get_state()
    assert np.max(np.abs(st["x"][0] - x0)) < 0.05 and np.max(np.abs(st["v"])) < 1e-3  # settles where the command timed out


def test_set_mass_rescales_row_two_and_inertia():
    s = one("f550")
    p0 = s.get_params(0)
    s.set_mass(3.0)
    p1 = s.get_params(0)
    assert p1.mass == 3.0
    assert np.allclose(np.array(p1.allocation_matrix[16:22]), np.array(p0.allocation_matrix[16:22]) * 3.0 / 2.3, rtol=1e-15)
    assert list(p1.allocation_matrix[:16]) == list(p0.allocation_matrix[:16]) and list(p1.allocation_matrix[24:]) == list(p0.allocation_matrix[24:])
    assert np.isclose(p1.J[8], 3.0 * 0.27 * 0.27 / 2.0) and np.isclose(p1.J[0], 3.0 * (3 * 0.27 ** 2 + 0.1 ** 2) / 12.0)

"""The persistent TMA-staged stepping kernel (`uav_step_staged_kernel`, csrc/step_kernel.cuh) after the edits that change what it
takes by value or stages, at batch sizes where it runs (58,001 UAVs: 454 tiles, the last one holds 17):

  * edited parameters, live rate integrals, external moments, feed-forwards and dt changes, against the CPU oracle;
  * a full inertia tensor against a long-double integration of Euler's equations (tests/test_full_inertia.py), and in closed loop
    against the oracle;
  * mrsb_run's tick graph, which holds the kernel's arguments by value, across changes of mode, dt, K, gains, parameters, moment
    and ground height;
  * a bucketed batch in which one bucket is edited whole, one partly (beyond its first tile) and one given a full J;
  * parameter-set collection followed by a staged launch.

With collisions off the UAVs are independent, so the oracle side is a sample of the batch built with the same spawn, commands and
edits (`sample`: every 97th UAV, both sides of the first tile boundaries and the partial last tile).  mrsb_get_step_info reports the
last bucket launched, so bucketed tests assert the staged launch of the highest airframe type.
"""
import os

import numpy as np
import pytest

from helpers import TOL, rand
from oracle import binding as O
from test_full_inertia import DT, L_DRIFT_TOL, OMEGA_TOL, STEPS, angular_momentum, euler_rk4, euler_states, free_body_airframe, full_inertia
from test_staged_parity_gpu import DT_PHASES, THREADS, af, big_grid, commands, edited_airframe, setup_flight, spawn_of

pytestmark = pytest.mark.gpu

MODES = [O.ACTUATOR_CMD, O.VELOCITY_HDG_RATE_CMD, O.VELOCITY_HDG_CMD, O.POSITION_CMD]
NM = {"x500": 4, "f550": 6, "naki": 8}
GAINS = {"rate": [4.2, 0.045, 0.6], "attitude": [6.5, 0.06, 0.05, 9.0, 1.2], "velocity": [2.2, 0.06, 0.05, 4.5], "position": [1.8, 0.12, 0.25, 5.0]}


def sample(n, step=97):
    """UAVs the oracle flies: every `step`-th, both sides of the first two tile boundaries, and the partial last tile."""
    last = (n - 1) // 128 * 128
    return np.unique(np.concatenate([np.arange(0, n, step), [127, 128, 129, 255, 256], np.arange(last - 2, n)])).astype(np.int32)


def sel(mask):
    return np.flatnonzero(mask).astype(np.int32)


class Env:
    """MRSB_* switches for the handles created inside the block (MRSB_NO_STAGING is read per launch)."""

    def __init__(self, **flags):
        self.flags = {k: v for k, v in flags.items() if v}

    def __enter__(self):
        for k in ("MRSB_NO_STAGING", "MRSB_NO_BUCKETS"):
            os.environ.pop(k, None)
        os.environ.update({k: "1" for k in self.flags})

    def __exit__(self, *exc):
        for k in ("MRSB_NO_STAGING", "MRSB_NO_BUCKETS"):
            os.environ.pop(k, None)


def assert_staged(b, mode, nm):
    info = b.step_info()
    assert info["variant"] == "staged" and info["mode"] == mode and info["n_motors"] == nm, info


def assert_same(a, b, what):
    for key in a:
        assert np.array_equal(a[key], b[key], equal_nan=True), f"{what}: {key} differs"


def assert_vs_oracle(orc, sg, mode, what):
    """Closed-loop modes within helpers.TOL; open-loop ActuatorCmd flight tumbles, so x, v and omega are compared relative to the
    excursion as in test_c5_actuator_cmd_staged_10s."""
    so = orc.get_state()
    if mode == O.ACTUATOR_CMD:
        for k in ("x", "v", "omega"):
            scale = 1.0 + np.max(np.abs(so[k]))
            assert np.max(np.abs(so[k] - sg[k])) <= 1e-7 * scale, f"{what}: {k}"
        assert np.max(np.abs(so["motor_rpm"] - sg["motor_rpm"])) <= 1e-5, f"{what}: motor_rpm"
        return
    bad = []
    for k, t in TOL.items():
        d = float(np.max(np.abs(so[k] - sg[k])))
        if not d <= t:
            bad.append(f"{k}: {d:.3e} > {t:.1e}")
    assert not bad, f"{what}: " + "; ".join(bad)


# ---- B: the edited flights of test_staged_equals_direct_bit_for_bit against the oracle ------------------------------------------
# The 8-motor edited flight is left to the bit-for-bit comparison: the naki, edited to 8.5 kg, flies with saturated motors, and at
# dt = 0.02 its rate loop is close enough to instability that ulp-level differences grow past helpers.TOL within 2 s (measured on a
# B200: omega 1.2e-8, motor_rpm 1.9e-5 after the 0.02 phase, the same for K = 1 and K = 10; 0.01 and 0.005 stay within 1e-10).
@pytest.mark.parametrize("frame,k", [("x500", 1), ("f550", 10)])
@pytest.mark.parametrize("mode", MODES)
def test_edited_staged_flight_vs_oracle(frame, k, mode):
    """setup_flight(..., "edited") — set_params with a full J, every gain with ki != 0, moments, feed-forwards — then 2 s at
    dt = 0.01, 1 s at 0.005 and 2 s at 0.02 on the staged kernel; a sample against the oracle."""
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 58001
    pick = sample(n)
    xyz, hdg = spawn_of(n)
    a = af(frame, ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=True)
    gpu = UavBatch([a], spawn_xyz=xyz, spawn_heading=hdg, n=n)
    orc = O.OracleSwarm([a], spawn_xyz=xyz[pick], spawn_heading=hdg[pick], n=len(pick))
    setup_flight(gpu, np.arange(n), n, frame, mode, "edited")
    setup_flight(orc, pick, n, frame, mode, "edited")
    for dt, seconds in zip(DT_PHASES, (2.0, 1.0, 2.0)):
        launches = int(round(seconds / dt / k))
        for _ in range(launches):
            gpu.make_step(dt, k)
        assert_staged(gpu, mode, NM[frame])
        orc.make_step(dt, launches * k, n_threads=THREADS)
    assert_vs_oracle(orc, gpu.get_full_state(pick), mode, f"edited {frame} flight, K = {k}")


# ---- C: a full inertia tensor ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 10])
def test_full_inertia_follows_eulers_equations_staged_and_direct(k):
    """Motors at 0 RPM, external moments only (tests/test_full_inertia.py): the body rates of the staged kernel
    (<4, ACTUATOR, K>) after 10 s against the long-double RK4 of Euler's equations, world-frame angular momentum conserved with
    zero moment, and the direct kernel identical in every bit."""
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 58001
    J = full_inertia()
    pick = sample(n)
    w0, tau = euler_states(J, np.arange(n))
    ref = euler_rk4(J, w0[pick], tau[pick])
    # the tolerance follows the rounding amplification of these very states (module docstring of test_full_inertia.py)
    tol = max(OMEGA_TOL, 5.0 * np.max(np.abs(euler_rk4(J, w0[pick], tau[pick], dtype=np.float64) - ref)))
    out = {}
    for staging in (True, False):
        with Env(MRSB_NO_STAGING=not staging):
            b = UavBatch([free_body_airframe(J)], spawn_xyz=big_grid(n, 100.0), spawn_heading=rand(6, 0, n, -3, 3), n=n)
            b.set_state(omega=w0)
            b.set_external_moment(tau)
            b.set_input(O.ACTUATOR_CMD, np.zeros((n, 8)))
            L0 = angular_momentum(b.get_full_state(pick), J)
            for _ in range(STEPS // k):
                b.make_step(DT, k)
            info = b.step_info()
            assert info["variant"] == ("staged" if staging else "direct") and info["mode"] == O.ACTUATOR_CMD, info
            out[staging] = b.get_full_state()
            out[staging]["crashed"] = b.has_crashed()
            b.close()
    assert_same(out[False], out[True], "staged vs direct kernel")
    s = {key: v[pick] for key, v in out[True].items()}
    assert np.all(s["motor_rpm"] == 0.0)
    d = float(np.max(np.abs(s["omega"] - ref)))
    assert d <= tol, f"omega differs from Euler's equations by {d:.3e} rad/s (tolerance {tol:.1e})"
    zero = ~tau[pick].any(axis=1)
    L = angular_momentum(s, J)
    drift = np.max(np.linalg.norm(L - L0, axis=1)[zero] / np.linalg.norm(L0, axis=1)[zero])
    assert drift <= L_DRIFT_TOL, f"world-frame angular momentum drifted by {drift:.3e}"


@pytest.mark.parametrize("n,variant", [(3000, "direct"), (58001, "staged")])
def test_full_inertia_closed_loop_vs_oracle(n, variant):
    """set_params with a full J for the whole batch, VelocityHdgCmd, 5 s: a sample against the oracle, on the direct kernel
    (3,000 UAVs) and on the staged kernel (58,001)."""
    from mrs_multirotor_simulator_b200 import UavBatch

    pick = sample(n)
    xyz, hdg = big_grid(n, 3.0), rand(8, 0, n, -3, 3)
    a = af("x500", ground_enabled=True, ground_z=0.0)
    gpu = UavBatch([a], spawn_xyz=xyz, spawn_heading=hdg, n=n)
    orc = O.OracleSwarm([a], spawn_xyz=xyz[pick], spawn_heading=hdg[pick], n=len(pick))
    cmd = commands(O.VELOCITY_HDG_CMD, n, seed=8)
    for s, g in ((gpu, np.arange(n)), (orc, pick)):
        s.set_params(edited_airframe("x500"))
        s.set_input(O.VELOCITY_HDG_CMD, cmd[g])
    for _ in range(500):
        gpu.make_step(0.01)
    orc.make_step(0.01, 500, n_threads=THREADS)
    info = gpu.step_info()
    assert info["variant"] == variant and info["mode"] == O.VELOCITY_HDG_CMD, info
    assert_vs_oracle(orc, gpu.get_full_state(pick), O.VELOCITY_HDG_CMD, f"full J, {variant} kernel")


# ---- D: the tick graph at staged size ------------------------------------------------------------------------------------------
def test_tick_graph_at_staged_size_follows_every_change():
    """Handle `a` issues make_step + handle_collisions, handle `b` calls mrsb_run, 25 ticks per block; between blocks both get
    the same change: the four staged modes in turn, a subset command (mixed modes: the direct kernel inside the graph), a
    whole-batch command again, dt, K, gains, set_params, the first external moment, set_ground_z.  After every block: pair lists,
    forces, crash flags and the full state bit for bit, and `b`'s last stepping launch staged wherever the batch is uniform."""
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 58001
    f550 = af("f550", ground_enabled=True, ground_z=0.0)
    spawn = big_grid(n, 4.0, pitch=2.0) + np.stack([rand(4, 0, n, -0.2, 0.2), rand(4, 1, n, -0.2, 0.2), rand(4, 2, n, -0.5, 0.5)], axis=1)
    a, b = UavBatch([f550], spawn_xyz=spawn, n=n), UavBatch([f550], spawn_xyz=spawn, n=n)
    for s in (a, b):
        s.set_collisions(True, False, 100.0)
        s.set_pair_capacity(16 * n)
    some = np.arange(0, n, 7, dtype=np.int32)
    third = np.arange(1, n, 3, dtype=np.int32)
    pos = np.concatenate([spawn[:, :2] + np.stack([rand(9, 0, n, -2, 2), rand(9, 1, n, -2, 2)], axis=1), rand(9, 2, n, 3, 6)[:, None],
                          rand(9, 3, n, -3, 3)[:, None]], axis=1)
    gains = lambda s: [s.set_controller_params(w, v) for w, v in GAINS.items()]
    # (what, change, dt, K, uniform mode afterwards or None for a mixed batch)
    blocks = [
        ("velocity_hdg_rate", lambda s: s.set_input(O.VELOCITY_HDG_RATE_CMD, commands(O.VELOCITY_HDG_RATE_CMD, n, 12)), 0.01, 1, O.VELOCITY_HDG_RATE_CMD),
        ("velocity_hdg", lambda s: s.set_input(O.VELOCITY_HDG_CMD, commands(O.VELOCITY_HDG_CMD, n, 13)), 0.01, 1, O.VELOCITY_HDG_CMD),
        ("position", lambda s: s.set_input(O.POSITION_CMD, pos), 0.01, 1, O.POSITION_CMD),
        ("actuator", lambda s: s.set_input(O.ACTUATOR_CMD, 0.5 + 0.1 * commands(O.ACTUATOR_CMD, n, 14)), 0.01, 1, O.ACTUATOR_CMD),
        ("subset command", lambda s: s.set_input(O.VELOCITY_HDG_RATE_CMD, commands(O.VELOCITY_HDG_RATE_CMD, n, 15)[some], idx=some), 0.01, 1, None),
        ("whole batch again", lambda s: s.set_input(O.POSITION_CMD, pos), 0.01, 1, O.POSITION_CMD),
        ("dt", lambda s: None, 0.005, 1, O.POSITION_CMD),
        ("K", lambda s: None, 0.005, 4, O.POSITION_CMD),
        ("gains", gains, 0.005, 4, O.POSITION_CMD),
        ("set_params", lambda s: s.set_params(edited_airframe("f550")), 0.005, 4, O.POSITION_CMD),
        ("first external moment", lambda s: s.set_external_moment(np.stack([rand(9, 4, len(third), -0.02, 0.02), rand(9, 5, len(third), -0.02, 0.02),
                                                                              rand(9, 6, len(third), -0.01, 0.01)], axis=1), idx=third), 0.005, 4, O.POSITION_CMD),
        ("set_ground_z", lambda s: s.set_ground_z(0.3), 0.005, 4, O.POSITION_CMD),
    ]
    total = 0
    for what, change, dt, k, mode in blocks:
        for s in (a, b):
            change(s)
        for _ in range(25):
            a.make_step(dt, k)
            a.handle_collisions()
        b.run(dt, 25, k)
        pa, pb = a.get_collision_pairs(), b.get_collision_pairs()
        assert np.array_equal(pa, pb), what
        total += len(pa)
        assert np.array_equal(a.get_force(), b.get_force()), what
        assert np.array_equal(a.has_crashed(), b.has_crashed()), what
        assert_same(a.get_full_state(), b.get_full_state(), f"mrsb_run vs separate calls after '{what}'")
        info = b.step_info()
        if mode is None:
            assert info["variant"] == "direct", (what, info)
        else:
            assert info["variant"] == "staged" and info["mode"] == mode and info["n_motors"] == 6, (what, info)
    assert total > 0
    assert b.counters()["steps"] == a.counters()["steps"] and b.counters()["collision_passes"] == a.counters()["collision_passes"]


# ---- E: partial edits of a bucketed batch --------------------------------------------------------------------------------------
PER_TYPE = 58001


def _bucketed_types():
    return [af("x500", ground_enabled=True), af("f550", ground_enabled=True), af("naki", ground_enabled=True)]


def _bucketed_setup(s, gidx, n):
    """x500 / f550 / naki interleaved by index.  Type 0: new gains for all of its UAVs (its bucket keeps one set, a new one).
    Type 1: set_mass on some UAVs past its bucket's first tile (the bucket becomes mixed).  Type 2: set_params with a full J for
    all of its UAVs."""
    t, rank = gidx % 3, gidx // 3
    s.set_input(O.VELOCITY_HDG_RATE_CMD, commands(O.VELOCITY_HDG_RATE_CMD, n, 17)[gidx])
    for which, v in GAINS.items():
        s.set_controller_params(which, v, idx=sel(t == 0))
    edited = sel((t == 1) & (rank >= 200) & (rank % 7 == 3))
    s.set_mass(2.3 * (1.0 + 0.05 * (1 + rank[edited] % 3)), idx=edited)
    s.set_params(edited_airframe("naki"), idx=sel(t == 2))


def _bucketed_flight(**env):
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 3 * PER_TYPE
    with Env(**env):
        b = UavBatch(_bucketed_types(), type_of_uav=(np.arange(n) % 3).astype(np.int32), spawn_xyz=big_grid(n, 2.0), n=n)
        _bucketed_setup(b, np.arange(n), n)
        for _ in range(300):
            b.make_step(0.01)
        info = b.step_info()
        out = b.get_full_state()
        out["crashed"] = b.has_crashed()
        out["mass"] = np.array([b.get_params(int(i)).mass for i in range(1, n, 3 * 97)])
        b.close()
    return out, info


def test_partial_edits_of_a_bucketed_batch():
    """3 x 58,001 UAVs, 3 s of VelocityHdgRateCmd: bit for bit equal with MRSB_NO_STAGING=1 and with MRSB_NO_BUCKETS=1, the naki
    bucket (the last one launched) staged, and a sample of every airframe against the oracle."""
    n = 3 * PER_TYPE
    out, info = _bucketed_flight()
    assert info["variant"] == "staged" and info["n_motors"] == 8 and info["mode"] == O.VELOCITY_HDG_RATE_CMD, info
    for env in ("MRSB_NO_STAGING", "MRSB_NO_BUCKETS"):
        other, info_o = _bucketed_flight(**{env: True})
        assert info_o["variant"] == "direct", (env, info_o)
        assert_same(out, other, f"bucketed vs {env}=1")
    ranks = sample(PER_TYPE)
    pick = np.sort(np.concatenate([3 * ranks + t for t in range(3)])).astype(np.int32)
    xyz = big_grid(n, 2.0)
    orc = O.OracleSwarm(_bucketed_types(), type_of_uav=(pick % 3).astype(np.int32), spawn_xyz=xyz[pick], n=len(pick))
    _bucketed_setup(orc, pick, n)
    orc.make_step(0.01, 300, n_threads=THREADS)
    assert_vs_oracle(orc, {k: out[k][pick] for k in TOL}, O.VELOCITY_HDG_RATE_CMD, "bucketed batch with partial edits")


# ---- F: parameter-set collection before a staged launch ------------------------------------------------------------------------
def _collected_flight(s, gidx, n, fly):
    """80 distinct masses (81 sets: more than 32), 1 s of flight on the direct kernel; then one airframe and one mass for all, so
    the unreferenced sets are collected and the one left renumbered, and 2 s on the staged kernel.  (set_mass alone cannot bring
    the batch back to one set: it rescales the yaw row of the allocation matrix by new / old mass (ROSW:1028-1080), which keeps
    ulp-level traces of the old mass.)"""
    s.set_input(O.VELOCITY_HDG_CMD, commands(O.VELOCITY_HDG_CMD, n, 19)[gidx])
    s.set_mass(1.6 + 0.01 * (gidx % 80))
    fly(100)
    s.set_params(af("x500", ground_enabled=True))
    s.set_mass(2.2)
    s.set_controller_params("rate", GAINS["rate"])
    fly(200)


def test_set_collection_then_staged_launch():
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 58001
    x500 = af("x500", ground_enabled=True)
    xyz = big_grid(n, 2.0)
    out = {}
    for staging in (True, False):
        with Env(MRSB_NO_STAGING=not staging):
            b = UavBatch([x500], spawn_xyz=xyz, n=n)
            infos = []

            def fly(steps):
                for _ in range(steps):
                    b.make_step(0.01)
                infos.append(b.step_info())

            _collected_flight(b, np.arange(n), n, fly)
            assert infos[0]["variant"] == "direct", infos
            if staging:
                assert infos[1]["variant"] == "staged" and infos[1]["mode"] == O.VELOCITY_HDG_CMD, infos
            out[staging] = b.get_full_state()
            out[staging]["crashed"] = b.has_crashed()
            assert {b.get_params(int(i)).mass for i in range(0, n, 1000)} == {2.2}
            b.close()
    assert_same(out[False], out[True], "staged vs direct kernel after set collection")
    pick = sample(n)
    orc = O.OracleSwarm([x500], spawn_xyz=xyz[pick], n=len(pick))
    _collected_flight(orc, pick, n, lambda steps: orc.make_step(0.01, steps, n_threads=THREADS))
    assert_vs_oracle(orc, {k: out[True][k][pick] for k in TOL}, O.VELOCITY_HDG_CMD, "after set collection")

"""The restated oracle (oracle/uav_oracle.hpp) against the reference's OWN UavSystem sources.

oracle/_ref/libref_uavsystem.so is uav_system.hpp + multirotor_model.hpp + controllers/*.hpp of the
reference, compiled unmodified from the reference tree's include/; only Eigen and Boost.odeint (absent
from the image) are replaced by the stand-ins under oracle/shim.  Both sides follow the same Eigen
evaluation rules, so the comparison is BIT-EXACT: any difference in dispatch, gains, clamps,
patches, NaN guards or scalar formulae between the restatement and the reference's code shows up
as a non-zero difference.  CPU only; the prebuilt library travels to the GPU box, where
tests/test_ref_uavsystem_gpu.py compares the CUDA path with it directly.

Without that library (the repository does not contain the reference's sources) every observation the
tests make of the reference side, PIDController results and default parameters included, is checked
against its stored digest (tests/golden/ref_uavsystem_digests.json, helpers.StoredResults).
"""
import os

import numpy as np
import pytest

from helpers import StoredResults, grid_spawn, rand
from mrs_multirotor_simulator_b200.airframes import airframe
from oracle import binding as O
from test_step_parity import ALL_MODES, _commands

FIELDS = ("x", "v", "R", "omega", "motor_rpm", "v_prev", "imu")
STORED = StoredResults(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_uavsystem_digests.json"))
Ref = STORED.swarm()
ref_lib = O.refsys_lib if STORED.mode != "check" else O.lib


@pytest.fixture(scope="module", autouse=True)
def _stored_results():
    yield from STORED.module()


@pytest.fixture(autouse=True)
def _observations(request):
    yield from STORED.run(request.node.name)


def pair(types, n, type_of_uav=None, spawn=None, heading=None):
    spawn = grid_spawn(n, z=10.0) if spawn is None else np.asarray(spawn, dtype=np.float64)
    heading = np.zeros(n) if heading is None else heading
    kw = dict(type_of_uav=type_of_uav, spawn_xyz=spawn, spawn_heading=heading, n=n)
    return O.OracleSwarm(types, **kw), Ref(types, **kw)


def assert_identical(orc, ref, what="", pid=True):
    so, sr = orc.get_state(), ref.get_state()
    for k in FIELDS:
        assert np.array_equal(so[k], sr[k], equal_nan=True), f"{what}: {k} differs by {np.nanmax(np.abs(so[k] - sr[k])):.3e}"
    if pid:
        for i in range(0, orc.n, max(1, orc.n // 8)):
            assert np.array_equal(orc.get_pid_state(i), ref.get_pid_state(i)), f"{what}: PID state of UAV {i}"


def both(orc, ref, fn):
    fn(orc)
    fn(ref)


# ------------------------------------------------------------------ every mode, every airframe
@pytest.mark.parametrize("frame", ["x500", "f550", "naki"])
@pytest.mark.parametrize("mode", ALL_MODES)
def test_every_mode_10s_bit_exact(mode, frame):
    n = 32
    orc, ref = pair([airframe(frame)], n, heading=rand(3, 0, n, -3, 3))
    cmd = _commands(mode, n)
    both(orc, ref, lambda s: s.set_input(mode, cmd))
    assert_identical(orc, ref, "spawn")
    for chunk in range(4):
        both(orc, ref, lambda s: s.make_step(0.01, 250))
        assert_identical(orc, ref, f"mode {mode} {frame} t={2.5 * (chunk + 1)} s")


def test_c1_hover_to_waypoint_and_golden_fixture():
    """BASELINE config 1 from the compiled reference == the committed fixture == the oracle."""
    import json

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c1_position_x500.json")) as f:
        g = json.load(f)
    orc, ref = pair([airframe("x500")], 1, spawn=[g["spawn"]], heading=np.array([g["heading"]]))
    both(orc, ref, lambda s: s.set_input(O.POSITION_CMD, [g["cmd"]]))
    for smp in g["samples"]:
        both(orc, ref, lambda s: s.make_step(g["dt"], 200))
        st = ref.get_state()
        for k in ("x", "v", "R", "omega", "motor_rpm", "imu"):
            assert np.array_equal(st[k][0], np.array(smp[k])), (smp["t"], k)
    assert_identical(orc, ref, "C1")
    assert np.allclose(ref.get_state()["x"][0], [4.99966878, -2.99316222, 3.99492282], atol=1e-8)  # SURVEY App. D


def test_golden_modes_fixture_is_the_compiled_reference():
    import json

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "modes_2s.json")) as f:
        g = json.load(f)
    for c in g["cases"]:
        ref = Ref([airframe(c["frame"])], spawn_xyz=[g["spawn"]], spawn_heading=[g["heading"]], n=1)
        ref.set_input(c["mode_id"], [c["cmd"]])
        ref.make_step(c["dt"], c["steps"])
        st = ref.get_state()
        for k in ("x", "v", "R", "omega", "motor_rpm", "imu"):
            assert np.array_equal(st[k][0], np.array(c[k])), (c["frame"], c["mode"], k)


# ------------------------------------------------------------------ mixer
@pytest.mark.parametrize("frame", ["x500", "f550", "naki", "t650"])
def test_mixer_allocation_and_every_desaturation_branch(frame):
    # rows: no saturation | min<0 shift | max>1 rescale (throttle>0.01) | max>1 divide (throttle<=0.01) |
    #       both | non-finite and out-of-range values into MultirotorModel::setInput's clamp
    cg = np.array([[0.02, -0.01, 0.03, 0.55], [0.5, 0.0, 0.0, 0.3], [0.3, 0.2, 0.1, 0.9], [0.3, 0.2, 0.1, 0.005], [0.9, 0.9, 0.9, 0.9],
                   [0.0, 0.0, 0.0, 1.2], [-0.7, 0.6, -0.5, 0.2], [np.nan, 0.0, 0.0, 0.5], [0.1, np.inf, 0.0, 0.5], [0.0, 0.0, 0.0, -0.4]])
    n = len(cg)
    for desat in (1.0, 0.0):
        orc, ref = pair([airframe(frame)], n)
        assert np.array_equal(orc.get_mixer_allocation(0), ref.get_mixer_allocation(0))
        both(orc, ref, lambda s: s.set_controller_params("mixer", [desat]))
        both(orc, ref, lambda s: s.set_input(O.CONTROL_GROUP_CMD, cg))
        both(orc, ref, lambda s: s.make_step(0.01, 3))
        assert_identical(orc, ref, f"{frame} desaturation={desat}")


def test_actuator_clamp_and_non_finite_inputs():
    act = np.array([[0.5, 0.5, 0.5, 0.5, 0, 0, 0, 0], [-0.2, 1.7, 0.5, 0.5, 0, 0, 0, 0], [np.nan, np.inf, -np.inf, 0.5, 0, 0, 0, 0]])
    orc, ref = pair([airframe("x500")], 3)
    both(orc, ref, lambda s: s.set_input(O.ACTUATOR_CMD, act))
    both(orc, ref, lambda s: s.make_step(0.01, 20))
    assert_identical(orc, ref, "actuator clamp")
    assert np.all(np.isfinite(ref.get_state()["motor_rpm"]))


# ------------------------------------------------------------------ patches, feed-forwards, events
def test_ground_clamp_and_one_way_takeoff_patch():
    n = 16
    types = [airframe("x500", ground_enabled=True, ground_z=0.0), airframe("f550", takeoff_patch_enabled=True)]
    tou = (np.arange(n) % 2).astype(np.int32)
    spawn = grid_spawn(n, z=0.0)
    spawn[1::2, 2] = 3.0
    orc, ref = pair(types, n, tou, spawn)
    both(orc, ref, lambda s: s.make_step(0.01, 50))
    assert_identical(orc, ref, "idle")
    assert np.array_equal(ref.get_state()["x"][:, 2], spawn[:, 2])
    both(orc, ref, lambda s: s.set_input(O.VELOCITY_HDG_RATE_CMD, np.tile([0.0, 0.0, 1.0, 0.3], (n, 1))))
    both(orc, ref, lambda s: s.make_step(0.01, 500))
    assert_identical(orc, ref, "take-off")
    assert ref.get_params(1).takeoff_patch_enabled == 0 and orc.get_params(1).takeoff_patch_enabled == 0
    even = np.arange(0, n, 2)
    both(orc, ref, lambda s: s.set_input(O.VELOCITY_HDG_RATE_CMD, np.tile([0.0, 0.0, -1.5, 0.0], (len(even), 1)), idx=even))
    both(orc, ref, lambda s: s.make_step(0.01, 800))
    assert_identical(orc, ref, "landing")
    assert np.all(ref.get_state()["x"][even, 2] == 0.0)


def test_feedforwards_sticky_and_precedence():
    n = 16
    orc, ref = pair([airframe("x500")], n, spawn=grid_spawn(n, z=5.0))
    ffv, ffa = np.tile([0.5, -0.25, 0.1, 0.0], (n, 1)), np.tile([0.2, 0.1, -0.1, 0.4], (n, 1))
    q, h = np.arange(0, n, 4), np.arange(0, n, 2)
    for mode in (O.POSITION_CMD, O.VELOCITY_HDG_RATE_CMD, O.VELOCITY_HDG_CMD, O.ACCELERATION_HDG_CMD):
        cmd = _commands(mode, n)
        both(orc, ref, lambda s: s.set_input(mode, cmd))
        if mode == O.POSITION_CMD:
            both(orc, ref, lambda s: s.set_feedforward(3, ffv))        # velocity_hdg_rate
            both(orc, ref, lambda s: s.set_feedforward(0, ffa))        # acceleration_hdg_rate
            both(orc, ref, lambda s: s.set_feedforward(1, 2 * ffa[q], q))  # acceleration_hdg on a quarter
            both(orc, ref, lambda s: s.set_feedforward(2, -ffv[h], h))     # velocity_hdg on half
        both(orc, ref, lambda s: s.make_step(0.01, 250))
        assert_identical(orc, ref, f"feed-forward, mode {mode}")


def test_crash_unknown_input_force_and_moment():
    n = 8
    orc, ref = pair([airframe("x500")], n, spawn=grid_spawn(n, z=50.0))
    cmd = _commands(O.VELOCITY_HDG_CMD, n)
    both(orc, ref, lambda s: s.set_input(O.VELOCITY_HDG_CMD, cmd))
    both(orc, ref, lambda s: s.apply_force(np.tile([1.0, -2.0, 0.5], (n, 1))))
    both(orc, ref, lambda s: s.make_step(0.01, 100))
    both(orc, ref, lambda s: s.crash([1, 5]))
    both(orc, ref, lambda s: s.set_input(O.INPUT_UNKNOWN, None, [2]))
    both(orc, ref, lambda s: s.set_external_moment(np.tile([0.01, 0.0, -0.02], (2, 1)), [3, 4]))
    both(orc, ref, lambda s: s.make_step(0.01, 100))
    assert_identical(orc, ref, "crash / unknown / force / moment")
    assert list(ref.has_crashed()) == list(orc.has_crashed()) == [0, 1, 0, 0, 0, 1, 0, 0]
    assert np.array_equal(orc.get_force(), ref.get_force())


def test_controller_params_and_set_params_reset():
    n = 8
    orc, ref = pair([airframe("x500")], n, spawn=grid_spawn(n, z=5.0))
    cmd = _commands(O.POSITION_CMD, n)

    def gains(s):
        s.set_input(O.POSITION_CMD, cmd)
        s.set_controller_params("position", [1.5, 0.1, 0.1, 3.0], [0, 1, 2, 3])
        s.set_controller_params("velocity", [2.5, 0.04, 0.02, 3.0], [2, 3])
        s.set_controller_params("attitude", [5.0, 0.04, 0.02, 8.0, 0.8], [3, 4])
        s.set_controller_params("rate", [3.0, 0.03, 0.01], [4, 5])
        s.set_controller_params("mixer", [0.0], [5, 6])

    both(orc, ref, gains)
    both(orc, ref, lambda s: s.make_step(0.01, 200))
    assert_identical(orc, ref, "custom gains")
    heavy = airframe("x500", mass=2.6)
    both(orc, ref, lambda s: s.set_params(heavy, [0, 3, 7]))  # US:404-409: gains back to defaults, PIDs reset
    assert np.array_equal(ref.get_pid_state(0), np.zeros(24)) and np.array_equal(orc.get_pid_state(0), np.zeros(24))
    assert ref.get_params(0).mass == 2.6 and ref.get_params(1).mass == 2.0
    both(orc, ref, lambda s: s.make_step(0.01, 300))
    assert_identical(orc, ref, "after setParams")


def test_set_state_and_single_steps_from_perturbed_states():
    n = 64
    for frame in ("x500", "f550", "naki"):
        nm = airframe(frame)["n_motors"]
        orc, ref = pair([airframe(frame)], n, spawn=grid_spawn(n, z=5.0), heading=rand(7, 0, n, -3, 3))
        st = orc.get_state()
        v = np.stack([rand(7, 1, n, -2, 2), rand(7, 2, n, -2, 2), rand(7, 3, n, -1, 1)], axis=1)
        w = np.stack([rand(7, 4, n, -0.5, 0.5), rand(7, 5, n, -0.5, 0.5), rand(7, 6, n, -0.5, 0.5)], axis=1)
        R = st["R"] + 1e-3 * np.stack([rand(7, 30 + k, n, -1, 1) for k in range(9)], axis=1)  # slightly non-orthonormal
        rpm = np.zeros((n, 8))
        rpm[:, :nm] = np.stack([rand(7, 20 + m, n, 3000, 5000) for m in range(nm)], axis=1)
        for mode in ALL_MODES:
            both(orc, ref, lambda s: s.set_state(x=st["x"], v=v, R=R, omega=w, motor_rpm=rpm))
            cmd = _commands(mode, n)
            both(orc, ref, lambda s: s.set_input(mode, cmd))
            both(orc, ref, lambda s: s.make_step(0.01, 3))
            assert_identical(orc, ref, f"{frame} mode {mode} from a perturbed state", pid=False)


def test_degenerate_requests_hit_the_same_nan_guards():
    """Free fall faster than g asked for (sqrt of a negative thrust -> NaN throttle -> isfinite guard,
    MM:399-401), zero tilt vector, zero-norm force direction, singular R (NaN slopes scrubbed, MM:361-365;
    step rolled back, MM:228-233)."""
    n = 4
    orc, ref = pair([airframe("x500")], n)
    acc = np.array([[0.0, 0.0, -15.0, 0.2], [0.0, 0.0, -9.81, 0.0], [30.0, 0.0, -9.0, 0.0], [1.0, 1.0, 1.0, 0.0]])
    both(orc, ref, lambda s: s.set_input(O.ACCELERATION_HDG_RATE_CMD, acc))
    both(orc, ref, lambda s: s.make_step(0.01, 50))
    assert_identical(orc, ref, "acceleration requests below -g")
    tilt = np.array([[0.0, 0.0, 0.0, 0.1, 0.5], [1e-200, 0.0, 0.0, 0.0, 0.5], [0.0, 0.0, -1.0, 0.0, 0.5], [0.3, 0.1, 1.0, 2.0, 0.5]])
    both(orc, ref, lambda s: s.set_input(O.TILT_HDG_RATE_CMD, tilt))
    both(orc, ref, lambda s: s.make_step(0.01, 50))
    assert_identical(orc, ref, "degenerate tilt vectors")
    st = orc.get_state()
    R = st["R"].copy()
    R[0] = 0.0                       # singular: Cholesky stops at the first pivot
    R[1, 3:6] = R[1, 0:3]            # rank 2
    both(orc, ref, lambda s: s.set_state(x=st["x"], v=st["v"], R=R, omega=st["omega"], motor_rpm=st["motor_rpm"]))
    both(orc, ref, lambda s: s.make_step(0.01, 5))
    assert_identical(orc, ref, "singular rotation matrices", pid=False)


def test_pid_controller_is_the_reference_class():
    rng = np.random.default_rng(5)
    for _ in range(200):
        kp, kd, ki = rng.uniform(0, 5, 3)
        sat = rng.choice([-1.0, 0.5, 4.0])
        aw = rng.choice([-1.0, 0.1, 1.0])
        sa, sb = np.zeros(2), np.zeros(2)
        for _ in range(20):
            e, dt = rng.uniform(-2, 2), rng.choice([0.001, 0.01, 0.02])
            ra = O.lib().orc_pid_update(O._p(sa), kp, kd, ki, sat, aw, e, dt)
            rb = ref_lib().orc_pid_update(O._p(sb), kp, kd, ki, sat, aw, e, dt)
            STORED.observe(np.append(rb, sb))
            assert ra == rb and np.array_equal(sa, sb)


def test_header_default_model_params():
    a, b = O.OrcModelParams(), O.OrcModelParams()
    O.lib().orc_model_params_default(O.C.byref(a))
    ref_lib().orc_model_params_default(O.C.byref(b))
    b.ground_z = a.ground_z  # the reference's default constructor leaves ground_z uninitialised (multirotor_model.hpp:84)
    STORED.observe(b)
    assert bytes(a) == bytes(b)
    assert a.n_motors == 4 and a.mass == 2.0 and a.takeoff_patch_enabled == 1 and a.ground_enabled == 0


# ------------------------------------------------------------------ how much can Eigen's evaluation order matter?
def test_eigen_evaluation_order_sensitivity_is_far_below_the_tolerance():
    """The one thing the compiled reference cannot pin is Eigen's own summation order.  Build it with
    the alternative reading (packet-ordered contiguous 3-term reductions, coefficient-based
    matrix x fixed-vector products) and measure the end-state difference after 10 s of closed-loop
    flight: it stays >= 100x below the parity tolerance (helpers.TOL)."""
    if O.refsys_lib("vec") is None:
        pytest.skip("libref_uavsystem_vec.so not built")
    from helpers import TOL

    n = 32
    worst = {k: 0.0 for k in ("x", "v", "R", "omega", "motor_rpm")}
    for frame in ("x500", "f550", "naki"):
        for mode in (O.ATTITUDE_CMD, O.TILT_HDG_RATE_CMD, O.ACCELERATION_HDG_RATE_CMD, O.ACCELERATION_HDG_CMD, O.VELOCITY_HDG_RATE_CMD,
                     O.VELOCITY_HDG_CMD, O.POSITION_CMD):
            kw = dict(spawn_xyz=grid_spawn(n, z=10.0), spawn_heading=rand(3, 0, n, -3, 3), n=n)
            a = O.RefSwarm([airframe(frame)], flavour="default", **kw)
            b = O.RefSwarm([airframe(frame)], flavour="vec", **kw)
            cmd = _commands(mode, n)
            both(a, b, lambda s: s.set_input(mode, cmd))
            both(a, b, lambda s: s.make_step(0.01, 1000))
            sa, sb = a.get_state(), b.get_state()
            for k in worst:
                worst[k] = max(worst[k], float(np.max(np.abs(sa[k] - sb[k]))))
    assert any(v > 0 for v in worst.values()), "the two builds are supposed to differ in rounding"
    for k, v in worst.items():
        assert v <= TOL[k] / 100.0, (k, v)


# ------------------------------------------------------------------ randomised event sequences
@pytest.mark.parametrize("seed", range(12))
def test_random_event_sequences_bit_exact(seed):
    """Fuzz: a random sequence of API calls (commands of every mode with ordinary, extreme and non-finite
    payloads, feed-forwards, crashes, forces, moments, gains, setParams, state teleports) interleaved with
    steps of varying dt on a mixed 4/6/8-motor swarm — the restatement must track the reference's own code
    bit for bit through all of it."""
    rng = np.random.default_rng(1000 + seed)
    n = 12
    frames = ["x500", "f550", "naki", "t650"]
    types = [airframe(f, ground_enabled=bool(rng.integers(2)), ground_z=float(rng.uniform(-1, 1)), takeoff_patch_enabled=bool(rng.integers(2))) for f in frames]
    tou = rng.integers(0, len(types), n).astype(np.int32)
    spawn = np.stack([rng.uniform(-20, 20, n), rng.uniform(-20, 20, n), rng.uniform(0, 10, n)], axis=1)
    orc, ref = pair(types, n, tou, spawn, heading=rng.uniform(-3.2, 3.2, n))

    def payload(mode, k):
        width = O.STRIDE[mode]
        kind = rng.integers(6)
        if kind == 0:  # ordinary flight-like values
            p = _commands(mode, k, seed=int(rng.integers(1 << 30)))
        elif kind == 1:
            p = rng.uniform(-1, 1, (k, width))
        elif kind == 2:
            p = rng.uniform(-50, 50, (k, width))
        elif kind == 3:
            p = np.zeros((k, width))
        elif kind == 4:
            p = rng.uniform(-1e6, 1e6, (k, width))
        else:
            p = rng.uniform(-2, 2, (k, width))
            bad = rng.integers(0, 4, (k, width))
            p[bad == 0] = rng.choice([np.nan, np.inf, -np.inf, 0.0, -0.0])
        return np.ascontiguousarray(p, dtype=np.float64)

    for event in range(120):
        what = rng.integers(12)
        idx = np.sort(rng.choice(n, int(rng.integers(1, n + 1)), replace=False)).astype(np.int32)
        if what <= 3:
            mode = int(rng.choice(ALL_MODES))
            pl = payload(mode, len(idx))
            both(orc, ref, lambda s: s.set_input(mode, pl, idx=idx))
        elif what == 4:
            kind = int(rng.integers(4))
            pl = rng.uniform(-2, 2, (len(idx), 4))
            both(orc, ref, lambda s: s.set_feedforward(kind, pl, idx))
        elif what == 5:
            f = rng.uniform(-5, 5, (len(idx), 3))
            both(orc, ref, lambda s: s.apply_force(f, idx))
        elif what == 6:
            m = rng.uniform(-0.05, 0.05, (len(idx), 3))
            both(orc, ref, lambda s: s.set_external_moment(m, idx))
        elif what == 7:
            which = str(rng.choice(["mixer", "rate", "attitude", "velocity", "position"]))
            vals = {"mixer": [float(rng.integers(2))], "rate": rng.uniform(0, 6, 3), "attitude": rng.uniform(0, 8, 5),
                    "velocity": rng.uniform(0, 4, 4), "position": rng.uniform(0, 4, 4)}[which]
            both(orc, ref, lambda s: s.set_controller_params(which, vals, idx))
        elif what == 8 and rng.integers(3) == 0:
            both(orc, ref, lambda s: s.crash(idx[:1]))
        elif what == 9 and rng.integers(2) == 0:
            # setParams keeps the airframe's motor count here (the reference would index motors out of range otherwise)
            one = idx[:1]
            f = frames[int(tou[one[0]])]
            p = airframe(f, mass=float(airframe(f)["mass"] * rng.uniform(0.7, 1.4)), ground_enabled=bool(rng.integers(2)),
                         ground_z=float(rng.uniform(-1, 1)), takeoff_patch_enabled=bool(rng.integers(2)))
            both(orc, ref, lambda s: s.set_params(p, one))
        elif what == 10 and rng.integers(2) == 0:
            st = orc.get_state(idx)
            x = st["x"] + rng.uniform(-1, 1, st["x"].shape)
            v = rng.uniform(-3, 3, st["v"].shape)
            both(orc, ref, lambda s: s.set_state(idx=idx, x=x, v=v, R=st["R"], omega=st["omega"], motor_rpm=st["motor_rpm"]))
        elif what == 11:
            both(orc, ref, lambda s: s.set_input(O.INPUT_UNKNOWN, None, idx[:1]))
        dt = float(rng.choice([0.001, 0.004, 0.005, 0.01, 0.02]))
        k = int(rng.integers(1, 12))
        both(orc, ref, lambda s: s.make_step(dt, k))
        assert_identical(orc, ref, f"seed {seed} event {event} (kind {what})", pid=False)
        assert np.array_equal(orc.has_crashed(), ref.has_crashed())
    for i in range(n):
        assert np.array_equal(orc.get_pid_state(i), ref.get_pid_state(i), equal_nan=True), i

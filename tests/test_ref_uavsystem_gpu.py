"""The CUDA stepping path against the reference side of tests/test_ref_uavsystem.py: the reference's OWN
UavSystem sources (oracle/_ref/libref_uavsystem.so: uav_system.hpp, multirotor_model.hpp,
controllers/*.hpp compiled unmodified against the Eigen/odeint stand-ins of oracle/shim) where that
build is present.  Without it the restatement stands in, and every state and crash flag it hands these
tests must equal its stored digest (tests/golden/ref_uavsystem_gpu_digests.json, helpers.StoredResults),
so that the GPU is compared with fixed results, not with whatever the restatement computes today.
Same tolerances as against the restated oracle (helpers.TOL, DESIGN.md §5)."""
import os

import numpy as np
import pytest

from helpers import TOL, StoredResults, grid_spawn, rand
from oracle import binding as O
from test_step_parity import ALL_MODES, _commands, af

pytestmark = pytest.mark.gpu

STORED = StoredResults(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_uavsystem_gpu_digests.json"))
Ref = STORED.swarm()


@pytest.fixture(scope="module", autouse=True)
def _stored_results():
    yield from STORED.module()


@pytest.fixture(autouse=True)
def _observations(request):
    yield from STORED.run(request.node.name)


def make(types, tou, spawn, heading=None):
    from mrs_multirotor_simulator_b200 import UavBatch

    n = len(spawn)
    heading = np.zeros(n) if heading is None else heading
    ref = Ref(types, type_of_uav=tou, spawn_xyz=spawn, spawn_heading=heading, n=n)
    gpu = UavBatch(types, type_of_uav=tou, spawn_xyz=spawn, spawn_heading=heading, n=n, device=0)
    return ref, gpu


def check(ref, gpu, what, tol=TOL):
    sr, sg = ref.get_state(), gpu.get_full_state()
    bad = []
    for k, t in tol.items():
        assert np.all(np.isfinite(sr[k])), f"reference {k} not finite ({what})"
        d = float(np.max(np.abs(sr[k] - sg[k])))
        if not d <= t:
            bad.append(f"{k}: {d:.3e} > {t:.1e}")
    assert not bad, f"{what}: " + "; ".join(bad)


def test_c1_single_x500_position_cmd_10s():
    ref, gpu = make([af("x500")], None, np.array([[0.0, 0.0, 1.0]]))
    for s in (ref, gpu):
        s.set_input(O.POSITION_CMD, [[5.0, -3.0, 4.0, 1.0]])
    ref.make_step(0.005, 2000)
    for _ in range(2000):
        gpu.make_step(0.005)
    check(ref, gpu, "C1")


@pytest.mark.parametrize("frame", ["x500", "f550", "naki"])
@pytest.mark.parametrize("mode", [m for m in ALL_MODES if m not in (O.ACTUATOR_CMD, O.CONTROL_GROUP_CMD, O.ATTITUDE_RATE_CMD)])
def test_10s_closed_loop_modes(mode, frame):
    n = 64
    ref, gpu = make([af(frame)], None, grid_spawn(n, z=10.0), rand(3, 0, n, -3, 3))
    cmd = _commands(mode, n)
    for s in (ref, gpu):
        s.set_input(mode, cmd)
    ref.make_step(0.01, 1000, n_threads=4)
    if mode == O.VELOCITY_HDG_CMD:  # the K-fused launch too
        for _ in range(100):
            gpu.make_step(0.01, 10)
    else:
        for _ in range(1000):
            gpu.make_step(0.01)
    check(ref, gpu, f"mode {mode} {frame}")


@pytest.mark.parametrize("mode", [O.ACTUATOR_CMD, O.CONTROL_GROUP_CMD, O.ATTITUDE_RATE_CMD])
def test_open_loop_modes(mode):
    """Open loop in attitude: compare one second tightly, before the tumbling amplifies rounding."""
    n = 64
    ref, gpu = make([af("x500")], None, grid_spawn(n, z=10.0), rand(3, 0, n, -3, 3))
    cmd = _commands(mode, n)
    for s in (ref, gpu):
        s.set_input(mode, cmd)
    ref.make_step(0.01, 100)
    for _ in range(100):
        gpu.make_step(0.01)
    check(ref, gpu, f"mode {mode}")


def test_c5_mixed_airframes_and_events():
    """Mixed 4/6/8-motor swarm, ground plane, custom gains, feed-forward, crash, force — 6 s."""
    n = 96
    types = [af(f, ground_enabled=True, ground_z=0.0) for f in ("x500", "f550", "naki")]
    tou = (np.arange(n) % 3).astype(np.int32)
    ref, gpu = make(types, tou, grid_spawn(n, z=0.0))
    cmd = _commands(O.POSITION_CMD, n)
    for s in (ref, gpu):
        s.set_input(O.POSITION_CMD, cmd)
        s.set_controller_params("position", [1.5, 0.1, 0.1, 3.0], [0, 1, 2, 3])
    ref.set_feedforward(0, np.tile([0.2, 0.1, -0.1, 0.4], (n, 1)))
    gpu.set_feedforward("acceleration_hdg_rate", np.tile([0.2, 0.1, -0.1, 0.4], (n, 1)))
    ref.make_step(0.01, 300)
    for _ in range(300):
        gpu.make_step(0.01)
    check(ref, gpu, "climb")
    for s in (ref, gpu):
        s.crash([5, 6, 7])
        s.apply_force(np.tile([1.0, -2.0, 0.5], (n, 1)))
    ref.make_step(0.01, 300)
    for _ in range(300):
        gpu.make_step(0.01)
    check(ref, gpu, "crash + force")
    assert np.all(gpu.get_state()["x"][[5, 6, 7], 2] == 0.0)  # the crashed ones fell onto the ground plane


@pytest.mark.parametrize("seed", range(6))
def test_random_event_sequences(seed):
    """Fuzz with finite, flight-like payloads: random commands of every mode, feed-forwards, forces, moments,
    gains, crashes, unknown input and setParams between steps of varying dt on a mixed 4/6/8-motor swarm.
    After every event the CUDA state must be within tolerance of the reference side; it is then
    re-synchronised to it (set_state), so that the open-loop modes' instability does not accumulate."""
    rng = np.random.default_rng(2000 + seed)
    n = 16
    frames = ["x500", "f550", "naki", "t650"]
    types = [af(f, ground_enabled=bool(rng.integers(2)), ground_z=float(rng.uniform(-1, 0)), takeoff_patch_enabled=bool(rng.integers(2))) for f in frames]
    tou = rng.integers(0, len(types), n).astype(np.int32)
    spawn = np.stack([rng.uniform(-20, 20, n), rng.uniform(-20, 20, n), rng.uniform(1, 10, n)], axis=1)
    ref, gpu = make(types, tou, spawn, rng.uniform(-3.0, 3.0, n))
    ff_names = ["acceleration_hdg_rate", "acceleration_hdg", "velocity_hdg", "velocity_hdg_rate"]
    tol = {"x": 1e-9, "v": 1e-8, "R": 1e-9, "omega": 1e-6, "motor_rpm": 1e-5, "imu": 1e-4}
    for event in range(40):
        what = int(rng.integers(10))
        idx = np.sort(rng.choice(n, int(rng.integers(1, n + 1)), replace=False)).astype(np.int32)
        if what <= 3:
            mode = int(rng.choice(ALL_MODES))
            pl = _commands(mode, len(idx), seed=int(rng.integers(1 << 30)))
            for s in (ref, gpu):
                s.set_input(mode, pl, idx=idx)
        elif what == 4:
            kind = int(rng.integers(4))
            pl = rng.uniform(-1, 1, (len(idx), 4))
            ref.set_feedforward(kind, pl, idx)
            gpu.set_feedforward(ff_names[kind], pl, idx)
        elif what == 5:
            f = rng.uniform(-3, 3, (len(idx), 3))
            for s in (ref, gpu):
                s.apply_force(f, idx)
        elif what == 6:
            m = rng.uniform(-0.02, 0.02, (len(idx), 3))
            for s in (ref, gpu):
                s.set_external_moment(m, idx)
        elif what == 7:
            which = str(rng.choice(["mixer", "rate", "attitude", "velocity", "position"]))
            vals = {"mixer": [float(rng.integers(2))], "rate": rng.uniform(1, 5, 3), "attitude": rng.uniform(1, 8, 5),
                    "velocity": rng.uniform(0.5, 4, 4), "position": rng.uniform(0.5, 4, 4)}[which]
            for s in (ref, gpu):
                s.set_controller_params(which, vals, idx)
        elif what == 8:
            if rng.integers(2):
                for s in (ref, gpu):
                    s.crash(idx[:1])
            else:
                for s in (ref, gpu):
                    s.set_input(O.INPUT_UNKNOWN, None, idx[:1])
        else:
            one = idx[:1]
            f = frames[int(tou[one[0]])]
            p = af(f, mass=float(af(f)["mass"] * rng.uniform(0.8, 1.3)), ground_enabled=bool(rng.integers(2)), ground_z=float(rng.uniform(-1, 0)),
                   takeoff_patch_enabled=bool(rng.integers(2)))
            for s in (ref, gpu):
                s.set_params(p, one)
        dt = float(rng.choice([0.004, 0.005, 0.01]))
        k = int(rng.integers(1, 8))
        ref.make_step(dt, k)
        for _ in range(k):
            gpu.make_step(dt)
        sr, sg = ref.get_state(), gpu.get_full_state()
        for key, t in tol.items():
            assert np.all(np.isfinite(sr[key])), (seed, event, key)
            scale = 1.0 + float(np.max(np.abs(sr[key])))
            d = float(np.max(np.abs(sr[key] - sg[key])))
            assert d <= t * scale, f"seed {seed} event {event} (kind {what}) {key}: {d:.3e} > {t * scale:.1e}"
        assert np.array_equal(np.asarray(ref.has_crashed()), np.asarray(gpu.has_crashed()))
        gpu.set_state(x=sr["x"], v=sr["v"], R=sr["R"], omega=sr["omega"], motor_rpm=sr["motor_rpm"])

"""mrsb_run replays CUDA graphs that hold their launch arguments by value: the collision pass and the whole tick (stepping launch
+ pass), one per buffer parity.  A graph that outlived a change of any of them would replay the old values without any sign on the
device.  Here every setter that changes such an argument is called in the middle of an mrsb_run sequence, and handle `a` (mrsb_run,
graphs) must stay equal bit for bit to handle `b`, which makes the same calls one by one with MRSB_NO_GRAPH=1 (read per call: the
ungraphed list pass rebuilds on every pass, the plain full pass, no tick graph).

Two batches: a bucketed one of three airframes (one stepping launch per bucket inside the tick graph), and a uniform one of 58,001
UAVs (454 tiles, more than 148 SMs x 3 CTAs) on which the persistent staged kernel, which takes the parameter set by value, runs.
"""
import os

import numpy as np
import pytest

from helpers import rand
from oracle import binding as O
from test_staged_parity_gpu import af, commands, edited_airframe

pytestmark = pytest.mark.gpu

TICKS = 20


class NoGraph:
    def __enter__(self):
        os.environ["MRSB_NO_GRAPH"] = "1"

    def __exit__(self, *exc):
        os.environ.pop("MRSB_NO_GRAPH", None)


def spawn_of(n, seed):
    side = int(np.ceil(np.sqrt(n)))
    i = np.arange(n)
    grid = np.stack([1.3 * (i % side), 1.3 * (i // side), np.full(n, 4.0)], axis=1)
    return grid + np.stack([rand(seed, 0, n, -0.2, 0.2), rand(seed, 1, n, -0.2, 0.2), rand(seed, 2, n, -0.5, 0.5)], axis=1)


def snapshot(b, imu):
    out = b.get_state(fields=("x", "v", "R", "omega", "motor_rpm", "v_prev") + (("imu",) if imu else ()))
    out["force"] = b.get_force()
    out["crashed"] = b.has_crashed()
    out["pairs"] = b.get_collision_pairs()  # sorted by the library
    return out


@pytest.mark.parametrize("batch", ["bucketed", "uniform_staged"])
def test_graphs_follow_every_change_inside_run(batch):
    from mrs_multirotor_simulator_b200 import UavBatch

    seed = 23
    if batch == "bucketed":
        n, names = 6000, ["x500", "f550", "naki"]
        tou = (np.arange(n) * 7 % 3).astype(np.int32)
    else:
        n, names = 58001, ["f550"]
        tou = None
    types = [af(name, ground_enabled=True, ground_z=0.0) for name in names]
    of_type = [np.arange(n, dtype=np.int32) if tou is None else np.flatnonzero(tou == t).astype(np.int32) for t in range(len(names))]
    spawn = spawn_of(n, seed)
    a = UavBatch(types, type_of_uav=tou, spawn_xyz=spawn, spawn_heading=rand(seed, 3, n, -3, 3), n=n)
    b = UavBatch(types, type_of_uav=tou, spawn_xyz=spawn, spawn_heading=rand(seed, 3, n, -3, 3), n=n)
    assert (a.device_view().slot_of_uav is not None) == (batch == "bucketed")
    some = np.arange(2, n, 9, dtype=np.int32)
    third = np.arange(1, n, 3, dtype=np.int32)
    pos = np.concatenate([spawn[:, :2] + np.stack([rand(seed, 4, n, -1, 1), rand(seed, 5, n, -1, 1)], axis=1), rand(seed, 6, n, 3, 5)[:, None],
                          rand(seed, 7, n, -3, 3)[:, None]], axis=1)

    def gains_params_mass(s):
        s.set_controller_params("velocity", [2.2, 0.06, 0.05, 4.5])
        s.set_mass(1.6 + 0.01 * (np.arange(n) % 80))  # 80 new parameter sets: the device table grows (moves)
        for name, idx in zip(names, of_type):  # one set per airframe again: the others are collected, ids renumbered
            s.set_params(edited_airframe(name), idx=idx)
        s.set_controller_params("rate", [4.2, 0.045, 0.6])

    # (what, change, dt, K); every change is made on both handles before the block's ticks
    blocks = [
        ("start", lambda s: s.set_input(O.VELOCITY_HDG_RATE_CMD, commands(O.VELOCITY_HDG_RATE_CMD, n, 12)), 0.01, 1),
        ("crash on", lambda s: s.set_collisions(True, True, 100.0), 0.01, 1),
        ("new rebounce", lambda s: s.set_collisions(True, True, 40.0), 0.01, 1),
        ("crash off", lambda s: s.set_collisions(True, False, 40.0), 0.01, 1),
        ("pair capacity", lambda s: s.set_pair_capacity(24 * n), 0.01, 1),
        ("outputs off", lambda s: s.set_outputs(imu=False, positions=False), 0.01, 1),
        ("outputs on", lambda s: s.set_outputs(imu=True, positions=True), 0.01, 1),
        ("iterate without input off", lambda s: s.set_iterate_without_input(False), 0.01, 1),
        ("dt", lambda s: None, 0.005, 1),
        ("K", lambda s: None, 0.005, 3),
        ("mode", lambda s: s.set_input(O.POSITION_CMD, pos), 0.005, 3),
        ("subset command", lambda s: s.set_input(O.VELOCITY_HDG_CMD, commands(O.VELOCITY_HDG_CMD, n, 13)[some], idx=some), 0.005, 3),
        ("respawn", lambda s: s.respawn(spawn[some] + np.array([0.3, -0.3, 0.5]), rand(seed, 11, len(some), -3, 3), idx=some), 0.005, 3),
        ("whole batch again", lambda s: s.set_input(O.VELOCITY_HDG_CMD, commands(O.VELOCITY_HDG_CMD, n, 14)), 0.005, 3),
        ("gains, set_mass, set_params", gains_params_mass, 0.005, 3),
        ("first external moment", lambda s: s.set_external_moment(np.stack([rand(seed, 8, len(third), -0.02, 0.02), rand(seed, 9, len(third), -0.02, 0.02),
                                                                              rand(seed, 10, len(third), -0.01, 0.01)], axis=1), idx=third), 0.005, 3),
        ("iterate without input on", lambda s: s.set_iterate_without_input(True), 0.01, 1),
    ]
    for s in (a, b):
        s.set_collisions(True, False, 100.0)
        s.set_pair_capacity(16 * n)
    imu, pairs, crashed = True, 0, 0
    for what, change, dt, k in blocks:
        for s in (a, b):
            change(s)
        imu = {"outputs off": False, "outputs on": True}.get(what, imu)
        a.run(dt, TICKS, k)
        with NoGraph():
            for _ in range(TICKS):
                b.make_step(dt, k)
                b.handle_collisions()
        sa, sb = snapshot(a, imu), snapshot(b, imu)
        for key in sa:
            assert np.array_equal(sa[key], sb[key], equal_nan=True), f"after '{what}': {key} differs"
        pairs += len(sa["pairs"])
        crashed = max(crashed, int(sa["crashed"].sum()))
    if batch == "uniform_staged":
        assert b.step_info()["variant"] == "staged" and a.step_info()["variant"] == "staged"
    assert pairs > 0 and crashed > 0, (pairs, crashed)
    ca, cb = a.counters(), b.counters()
    assert (ca["steps"], ca["collision_passes"]) == (cb["steps"], cb["collision_passes"])
    a.close()
    b.close()

"""On a single-bucket handle whose state is larger than L2, the staged stepping kernel walks its tiles from the front on one
launch and from the back on the next (the parity of a device word per bucket, advanced by every such launch).  Results must not
depend on the direction: after any number of launches, and through mrsb_run's cached tick graph, the staged kernel equals the
direct kernel (`MRSB_NO_STAGING=1`) bit for bit — state, packed positions, forces, pair lists and the collision pass' counters —
and mrsb_get_sweep_launches shows that the direction did alternate (or, for bucketed and small batches, that it did not).

Sizes are chosen so that the tile count is not a multiple of the persistent grid and the last tile is partial."""
import os

import numpy as np
import pytest

from helpers import rand
from oracle import binding as O

pytestmark = pytest.mark.gpu

FIELDS = ("x", "v", "R", "omega", "motor_rpm", "v_prev", "imu")


def grid(n, pitch, z):
    side = int(np.ceil(np.sqrt(n)))
    i = np.arange(n)
    return np.stack([pitch * (i % side), pitch * (i // side), np.full(n, z)], axis=1).astype(np.float64)


def velocity_cmd(n, seed=7):
    return np.stack([rand(seed, 1, n, -2, 2), rand(seed, 2, n, -2, 2), rand(seed, 3, n, -1, 1), rand(seed, 4, n, -1, 1)], axis=1)


def fly(staging, frames, n, pitch, launches=0, run_calls=(), collisions=False):
    """One handle: `launches` make_step calls, then one mrsb_run call per entry of run_calls (ticks per call)."""
    import torch

    from mrs_multirotor_simulator_b200 import UavBatch, airframe

    if staging:
        os.environ.pop("MRSB_NO_STAGING", None)
    else:
        os.environ["MRSB_NO_STAGING"] = "1"
    try:
        types = [airframe(f) for f in frames]
        tou = (np.arange(n) % len(frames)).astype(np.int32) if len(frames) > 1 else None
        b = UavBatch(types, type_of_uav=tou, spawn_xyz=grid(n, pitch, 20.0), n=n)
        b.set_input(O.VELOCITY_HDG_RATE_CMD, velocity_cmd(n))
        if collisions:
            b.set_collisions(True, False, 100.0)
            b.set_pair_capacity(8 * n)  # every UAV of the dense grid touches its neighbours
        for _ in range(launches):
            b.make_step(0.01)
        for ticks in run_calls:
            b.run(0.01, ticks, 1, collisions)
        out = b.get_full_state()
        out["crashed"] = b.has_crashed()
        packed = torch.empty((n, 3), dtype=torch.float64).pin_memory()  # the packed positions the collision pass reads
        b.get_positions_async(packed.data_ptr())
        b.sync()
        out["packed_x"] = packed.numpy().copy()
        out["info"] = b.step_info()
        out["sweeps"] = b.sweep_launches()
        if collisions:
            out["force"] = b.get_force()
            out["pairs"] = b.get_collision_pairs()
            info = b.collision_info()
            out["collision_info"] = np.array([info["passes"], info["rebuilds"], info["crowded_uavs"]])
            out["counters"] = np.array([b.counters()["pairs"]])
        b.close()
        return out
    finally:
        os.environ.pop("MRSB_NO_STAGING", None)


def assert_same(direct, staged, alternating):
    """alternating: the number of staged launches of each bucket that must have swept with alternating direction"""
    assert direct["info"]["variant"] == "direct", direct["info"]
    assert staged["info"]["variant"] == "staged", staged["info"]
    assert direct["sweeps"] == [0] * len(alternating), direct["sweeps"]
    assert staged["sweeps"] == alternating, staged["sweeps"]
    for key in direct:
        if key in ("info", "sweeps"):
            continue
        assert np.array_equal(direct[key], staged[key], equal_nan=True), f"{key} differs between the staged and the direct kernel"
    assert np.all(np.isfinite(staged["x"]))


BIG = 4096 * 128 + 9  # 4097 tiles (the last holds 9 UAVs): ~180 MB of tile images per launch, more than L2


@pytest.mark.parametrize("launches", [1, 2, 3])
def test_both_sweep_directions_equal_direct(launches):
    """x500 over a persistent grid that does not divide the tiles; launches 2 and 3 sweep backward and forward again."""
    assert_same(fly(False, ["x500"], BIG, 4.0, launches), fly(True, ["x500"], BIG, 4.0, launches), [launches])


def test_state_that_fits_l2_sweeps_forward():
    """85,001 x500 (665 tiles, ~30 MB of tile images): nothing to gain from alternating — every launch sweeps forward."""
    n = 85001
    assert_same(fly(False, ["x500"], n, 4.0, 3), fly(True, ["x500"], n, 4.0, 3), [0])


def test_bucketed_batch_sweeps_forward():
    """x500 / f550 / naki interleaved: three buckets of 200,001 UAVs (1563 tiles each, partial last tile), three staged launches
    per tick.  Between two launches of a bucket the other two stream their state through L2: no bucket alternates."""
    n = 3 * 200001
    frames = ["x500", "f550", "naki"]
    assert_same(fly(False, frames, n, 4.0, 3), fly(True, frames, n, 4.0, 3), [0, 0, 0])


@pytest.mark.parametrize("run_calls", [(2,), (3,), (1, 2)])
def test_ticks_through_the_cached_graph(run_calls):
    """mrsb_run with collisions on a dense grid (0.6 m pitch: pairs every tick) after one make_step: 2 and 3 ticks in one call,
    and 1 + 2 in two calls (the second replays the graph the first captured) — both directions run inside the replayed graph."""
    direct = fly(False, ["x500"], BIG, 0.6, 1, run_calls, collisions=True)
    staged = fly(True, ["x500"], BIG, 0.6, 1, run_calls, collisions=True)
    assert len(staged["pairs"]) > 0
    assert_same(direct, staged, [1 + sum(run_calls)])

"""Pipelined node-loop I/O: mixed-mode command rows in (mrsb_set_input_rows_async), odometry | IMU | range rows out
(mrsb_get_observations_async).  Everything is checked bit for bit against a twin handle driven through the blocking calls:
rows after a "last occurrence wins" dedup go in through mrsb_set_input, one call per mode; sensor rows come out of
mrsb_pack_observations_device and positions out of mrsb_get_state."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from helpers import grid_spawn, rand
from oracle import binding as O
from test_cpp_facade import build
from test_sharded_gpu import exchange, make_shards
from test_step_parity import ALL_MODES, _commands

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STRIDE = {O.ACTUATOR_CMD: 8, O.ATTITUDE_CMD: 10, O.TILT_HDG_RATE_CMD: 5}  # every other payload mode: 4


def af(name, **kw):
    from mrs_multirotor_simulator_b200 import airframe

    return airframe(name, **kw)


def pinned(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


def pinned_zeros(*shape):
    import torch

    return torch.zeros(shape, dtype=torch.float64).pin_memory()


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def random_rows(rng, n, count, stride, seed):
    """`count` rows for random UAVs (repeats happen) in every mode whose row fits `stride` (actuator rows always: motors past the
    stride are 0), then three UAVs again with a different mode each — the last two of them a third time."""
    allowed = [m for m in ALL_MODES if m == O.ACTUATOR_CMD or STRIDE.get(m, 4) <= stride]
    idx = [int(i) for i in rng.integers(0, n, count)]
    modes = [int(m) for m in rng.choice(allowed, count)]
    again = [int(i) for i in rng.choice(np.unique(idx), 3, replace=False)]
    for e in again + again[1:]:
        prev = modes[len(idx) - 1 - idx[::-1].index(e)]
        idx.append(e)
        modes.append(allowed[(allowed.index(prev) + 1) % len(allowed)])
    idx, modes = np.array(idx), np.array(modes)
    rows = np.zeros((len(idx), stride))
    for m in allowed:
        sel = modes == m
        if sel.any():
            cmd = _commands(int(m), int(sel.sum()), seed=seed + int(m))
            rows[sel, :min(stride, cmd.shape[1])] = cmd[:, :stride]
    return idx.astype(np.int32), modes.astype(np.int32), rows


def dedup(idx, modes, rows):
    """The rows that win: the last one of every UAV (in first-appearance order of the winners, which does not matter)."""
    _, first_rev = np.unique(idx[::-1], return_index=True)
    keep = np.sort(len(idx) - 1 - first_rev)
    return idx[keep], modes[keep], rows[keep]


def set_blocking(b, idx, modes, rows, stride):
    """The twin's side: mrsb_set_input with the same stride, one call per mode, after the dedup."""
    from mrs_multirotor_simulator_b200._lib import check

    idx, modes, rows = dedup(idx, modes, rows)
    for m in np.unique(modes):
        i = np.ascontiguousarray(idx[modes == m], dtype=np.int32)
        r = np.ascontiguousarray(rows[modes == m], dtype=np.float64)
        check(b._L.mrsb_set_input(b.h, int(m), len(i), ptr(i), ptr(r), stride))


class RowCall:
    """The pinned host arrays of one mrsb_set_input_rows_async call, kept alive until the handle is synchronised."""

    def __init__(self, idx, modes, rows):
        self.idx, self.modes, self.rows = pinned(idx.astype(np.int32)), pinned(modes.astype(np.int32)), pinned(rows.astype(np.float64))
        self.stride = rows.shape[1]

    def send(self, b):
        b.set_input_rows_async(len(self.idx), self.idx.data_ptr(), self.modes.data_ptr(), self.rows.data_ptr(), self.stride)


def assert_same(a, b, what=""):
    a.sync()
    b.sync()
    fa, fb = a.get_full_state(), b.get_full_state()
    for k in fa:
        assert np.array_equal(fa[k], fb[k]), (what, k)
    assert np.array_equal(a.get_input_mode(), b.get_input_mode()), what
    # the stored commands, cached cos/sin of the heading, flags ("had a command") and modes: the snapshot records, header aside
    sa, sb = a.snapshot(), b.snapshot()
    sa.save()
    sb.save()
    assert sa.to_bytes()[48:] == sb.to_bytes()[48:], what
    sa.free()
    sb.free()


def bucketed_pair(n, seed, pitch=1.5):
    from mrs_multirotor_simulator_b200 import UavBatch

    types = [af("x500"), af("f550"), af("naki")]
    tou = np.random.default_rng(seed).integers(0, 3, n).astype(np.int32)
    spawn = grid_spawn(n, pitch=pitch, z=5.0)
    return [UavBatch(types, type_of_uav=tou, spawn_xyz=spawn, n=n) for _ in range(2)]


def test_rows_equal_blocking_calls_bit_for_bit():
    """A padded, bucketed batch of x500 / f550 / naki, 50 ticks with collisions; every tick a random set of rows of all the modes its
    stride allows (strides 10, 8, 5, 4: actuator rows shorter than 8 motors), with UAVs addressed two and three times in one call."""
    n = 1000
    a, b = bucketed_pair(n, 1, pitch=0.9)
    for s in (a, b):
        s.set_collisions(True, False, 100.0)
    rng = np.random.default_rng(2)
    calls, seen_modes, dup_modes, pairs = [], set(), 0, 0
    for t in range(50):
        stride = (10, 8, 5, 4)[t % 4]
        idx, modes, rows = random_rows(rng, n, int(rng.integers(20, 200)), stride, seed=100 * t)
        seen_modes |= set(modes.tolist())
        dup_modes += sum(len(set(modes[idx == u].tolist())) > 1 for u in np.unique(idx))
        calls.append(RowCall(idx, modes, rows))
        calls[-1].send(a)
        set_blocking(b, idx, modes, rows, stride)
        for s in (a, b):
            s.run(0.01, 1)
        p = a.get_collision_pairs()
        assert np.array_equal(p, b.get_collision_pairs()), t
        pairs += len(p)
    assert seen_modes == set(ALL_MODES) and dup_modes >= 50 and pairs > 0
    assert_same(a, b)


def test_rows_keep_a_uniform_batch_uniform():
    """58,001 x500: after one whole-batch VelocityHdgRate call, VelocityHdgRate rows every tick keep the staged kernel specialised for
    that mode; one row of another mode makes the batch per-UAV-mode; the next whole-batch call restores the specialisation."""
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 58001
    b = UavBatch([af("x500")], spawn_xyz=grid_spawn(n, z=5.0), n=n)
    whole = pinned(np.stack([rand(3, 1, n, -2, 2), rand(3, 2, n, -2, 2), rand(3, 3, n, 0, 2), rand(3, 4, n, -1, 1)], axis=1))
    b.set_input_async(O.VELOCITY_HDG_RATE_CMD, whole.data_ptr(), 4)
    rng = np.random.default_rng(4)
    calls = []
    for t in range(5):
        idx = rng.integers(0, n, 600).astype(np.int32)
        calls.append(RowCall(idx, np.full(len(idx), O.VELOCITY_HDG_RATE_CMD), _commands(O.VELOCITY_HDG_RATE_CMD, len(idx), seed=t)))
        calls[-1].send(b)
        b.make_step(0.01)
        info = b.step_info()
        assert info["variant"] == "staged" and info["mode"] == O.VELOCITY_HDG_RATE_CMD, (t, info)
    calls.append(RowCall(np.array([17]), np.array([O.POSITION_CMD]), np.array([[1.0, 2.0, 3.0, 0.5]])))
    calls[-1].send(b)
    b.make_step(0.01)
    assert b.step_info()["mode"] == -1
    b.set_input_async(O.VELOCITY_HDG_RATE_CMD, whole.data_ptr(), 4)
    b.make_step(0.01)
    info = b.step_info()
    assert info["variant"] == "staged" and info["mode"] == O.VELOCITY_HDG_RATE_CMD, info
    b.sync()
    assert np.all(b.get_input_mode() == O.VELOCITY_HDG_RATE_CMD)


@pytest.mark.parametrize("subset", [False, True])
def test_forty_ticks_enqueued_back_to_back(subset):
    """rows -> run -> positions -> observations for 40 ticks with no synchronisation, each tick with its own pinned buffers; after one
    sync every tick's downloads equal the blocking twin's positions and mrsb_pack_observations_device rows at that tick."""
    import torch

    n = 3000
    a, b = bucketed_pair(n, 5)
    sub = np.random.default_rng(6).permutation(n)[:700].astype(np.int32) if subset else None
    m = n if sub is None else len(sub)
    a.set_position_subset(sub)
    for s in (a, b):
        s.set_collisions(True, False, 100.0)
    rng = np.random.default_rng(7)
    calls, pos, obs, ref_pos, ref_obs = [], [], [], [], []
    dev = torch.zeros((n, 17), dtype=torch.float64, device="cuda")
    for t in range(40):
        idx, modes, rows = random_rows(rng, n, int(rng.integers(50, 400)), 10, seed=1000 + 10 * t)
        calls.append(RowCall(idx, modes, rows))
        pos.append(pinned_zeros(m, 3))
        obs.append(pinned_zeros(m, 17))
        calls[-1].send(a)
        a.run(0.01, 1)
        a.get_positions_async(pos[-1].data_ptr())
        a.get_observations_async(obs[-1].data_ptr())
    for t in range(40):
        set_blocking(b, calls[t].idx.numpy(), calls[t].modes.numpy(), calls[t].rows.numpy(), 10)
        b.run(0.01, 1)
        ref_pos.append(b.get_state(idx=sub, fields=("x",))["x"])
        b.pack_observations_device(dev.data_ptr(), 17)
        b.sync()
        ref_obs.append(dev.cpu().numpy()[sub if subset else slice(None)])
    a.sync()
    for t in range(40):
        assert np.array_equal(pos[t].numpy(), ref_pos[t]), t
        assert np.array_equal(obs[t].numpy(), ref_obs[t]), t
    assert_same(a, b)


def test_rows_revive_timed_out_uavs():
    """iterate_without_input off: UAVs stopped by an input timeout stay frozen until a row reaches them, exactly as with the blocking
    call; the ones no row reaches stay frozen."""
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 300
    a, b = [UavBatch([af("x500")], spawn_xyz=grid_spawn(n, z=5.0), n=n) for _ in range(2)]
    cmd = np.stack([rand(8, 1, n, -2, 2), rand(8, 2, n, -2, 2), rand(8, 3, n, 0, 2), rand(8, 4, n, -1, 1)], axis=1)
    timed_out = np.arange(0, n, 2, dtype=np.int32)
    for s in (a, b):
        s.set_iterate_without_input(False)
        s.set_input(O.VELOCITY_HDG_RATE_CMD, cmd)
        s.run(0.01, 20)
        s.timeout_input(timed_out)
        s.run(0.01, 10)
    frozen = a.get_full_state(timed_out)
    revived = timed_out[::3]
    idx = np.concatenate([revived, revived[:5]]).astype(np.int32)
    modes = np.concatenate([np.full(len(revived), O.POSITION_CMD), np.full(5, O.VELOCITY_HDG_CMD)])
    rows = np.concatenate([_commands(O.POSITION_CMD, len(revived), seed=9), _commands(O.VELOCITY_HDG_CMD, 5, seed=10)])
    call = RowCall(idx, modes, rows)
    call.send(a)
    set_blocking(b, idx, modes, rows, 4)
    for s in (a, b):
        s.run(0.01, 20)
    assert_same(a, b)
    still = np.setdiff1d(timed_out, revived)
    now = a.get_full_state(still)
    sel = np.searchsorted(timed_out, still)
    for k in frozen:
        assert np.array_equal(now[k], frozen[k][sel]), k
    assert not np.array_equal(a.get_state(revived)["x"], frozen["x"][np.searchsorted(timed_out, revived)])


def test_a_row_call_larger_than_the_staging_ring():
    """Small row calls and a whole-batch call in flight, then a row call of three times the swarm (every UAV addressed three times)
    that outgrows both staging rings: the same bits as the blocking twin."""
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 2000
    a, b = [UavBatch([af("f550")], spawn_xyz=grid_spawn(n, z=5.0), n=n) for _ in range(2)]
    rng = np.random.default_rng(11)
    calls = []
    whole = pinned(_commands(O.VELOCITY_HDG_CMD, n, seed=12))
    for t in range(6):
        if t == 2:
            a.set_input_async(O.VELOCITY_HDG_CMD, whole.data_ptr(), 4)
            b.set_input(O.VELOCITY_HDG_CMD, whole.numpy())
        idx, modes, rows = random_rows(rng, n, 10, 4, seed=200 + t)
        calls.append(RowCall(idx, modes, rows))
        calls[-1].send(a)
        set_blocking(b, idx, modes, rows, 4)
        for s in (a, b):
            s.run(0.01, 1)
    idx = np.concatenate([rng.permutation(n) for _ in range(3)]).astype(np.int32)
    modes = rng.choice(ALL_MODES, len(idx)).astype(np.int32)
    rows = np.zeros((len(idx), 10))
    for m in ALL_MODES:
        sel = modes == m
        c = _commands(m, int(sel.sum()), seed=300 + m)
        rows[sel, :c.shape[1]] = c
    calls.append(RowCall(idx, modes, rows))
    calls[-1].send(a)
    set_blocking(b, idx, modes, rows, 10)
    for t in range(3):
        idx, modes, rows = random_rows(rng, n, 10, 10, seed=400 + t)
        calls.append(RowCall(idx, modes, rows))
        calls[-1].send(a)
        set_blocking(b, idx, modes, rows, 10)
        for s in (a, b):
            s.run(0.01, 1)
    assert_same(a, b)


def test_refusals_leave_the_state_untouched():
    from mrs_multirotor_simulator_b200 import UavBatch
    from mrs_multirotor_simulator_b200._lib import MrsbError

    n = 64
    b = UavBatch([af("x500")], spawn_xyz=grid_spawn(n, z=5.0), n=n)
    b.set_input(O.VELOCITY_HDG_RATE_CMD, np.tile([0.5, 0.0, 0.1, 0.2], (n, 1)))
    b.make_step(0.01)
    s = b.snapshot()
    s.save()
    before = s.to_bytes()
    i1, m1, r10 = pinned(np.array([3], np.int32)), pinned(np.array([O.POSITION_CMD], np.int32)), pinned(np.ones((1, 10)))
    bad = [
        (1, pinned(np.array([n], np.int32)), m1, r10, 4),  # index past the end
        (2, pinned(np.array([0, -1], np.int32)), pinned(np.array([8, 8], np.int32)), pinned(np.ones((2, 4))), 4),  # negative index
        (1, i1, pinned(np.array([0], np.int32)), r10, 4),  # mode 0
        (1, i1, pinned(np.array([11], np.int32)), r10, 10),  # mode 11
        (2, pinned(np.array([1, 2], np.int32)), pinned(np.array([8, 4], np.int32)), pinned(np.ones((2, 5))), 5),  # attitude needs 10
        (1, i1, pinned(np.array([5], np.int32)), r10, 4),  # tilt needs 5
        (1, i1, m1, r10, 3),  # position needs 4
        (1, i1, pinned(np.array([1], np.int32)), r10, 0),  # actuators need >= 1
        (1, None, m1, r10, 4),
        (1, i1, None, r10, 4),
        (1, i1, m1, None, 4),
        (-1, i1, m1, r10, 4),
        (2 ** 31, i1, m1, r10, 4),  # refused before anything is read
    ]
    for k, (cnt, idx, modes, rows, stride) in enumerate(bad):
        with pytest.raises(MrsbError) as e:
            b.set_input_rows_async(cnt, *[None if x is None else x.data_ptr() for x in (idx, modes, rows)], stride)
        assert e.value.code == -1, k
    b.set_input_rows_async(0, None, None, None, 4)  # n == 0: a no-op
    b.sync()
    s.save()
    assert s.to_bytes() == before
    b.set_outputs(imu=False, positions=True)
    out = pinned_zeros(n, 17)
    with pytest.raises(MrsbError) as e:
        b.get_observations_async(out.data_ptr())
    assert e.value.code == -5
    with pytest.raises(MrsbError) as e:
        b.get_observations_async(None)
    assert e.value.code == -1


def test_sharded_rows_equal_the_unsharded_run():
    """Two handles on one GPU own the two halves of the swarm; each gets its own shard's rows (local indices, in the order of the
    whole call) and the result equals the unsharded handle fed the whole rows, bit for bit."""
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 1024
    t = af("f550", ground_enabled=True)
    spawn = grid_spawn(n, pitch=1.2, z=3.0)
    whole = UavBatch([t], spawn_xyz=spawn, n=n)
    shards = make_shards([t], None, spawn, (0, 512, 1024))
    for s in [whole] + shards:
        s.set_collisions(True, False, 100.0)
        s.set_pair_capacity(8 * n)
    rng = np.random.default_rng(13)
    calls = []
    for tick in range(30):
        idx, modes, rows = random_rows(rng, n, 150, 10, seed=500 + 10 * tick)
        calls.append(RowCall(idx, modes, rows))
        calls[-1].send(whole)
        for sh in shards:
            sel = (idx >= sh.shard_begin) & (idx < sh.shard_begin + sh.n)
            calls.append(RowCall(idx[sel] - sh.shard_begin, modes[sel], rows[sel]))
            calls[-1].send(sh)
        whole.make_step(0.01)
        whole.handle_collisions()
        for sh in shards:
            sh.make_step(0.01)
        exchange(shards)
        for sh in shards:
            sh.handle_collisions_gathered()
    whole.sync()
    sw, mw = whole.get_full_state(), whole.get_input_mode()
    for sh in shards:
        sh.sync()
        ss = sh.get_full_state()
        for k in sw:
            assert np.array_equal(sw[k][sh.shard_begin:sh.shard_begin + sh.n], ss[k]), k
        assert np.array_equal(mw[sh.shard_begin:sh.shard_begin + sh.n], sh.get_input_mode())


def node_commands(t, n):
    """tests/cpp/node_loop_async.cpp's commands(t): the same rows, the same arithmetic."""
    kinds = [O.VELOCITY_HDG_RATE_CMD, O.VELOCITY_HDG_CMD, O.POSITION_CMD, O.ACCELERATION_HDG_RATE_CMD]
    idx, modes, rows = [], [], []

    def add(i, m):
        idx.append(i)
        modes.append(kinds[m])
        if kinds[m] == O.POSITION_CMD:
            rows.append([2.0 * (i % 16) + 0.5, 2.0 * (i // 16) - 0.5, 3.0 + 0.25 * (t % 4), 0.3])
        elif kinds[m] == O.ACCELERATION_HDG_RATE_CMD:
            rows.append([0.2 * ((i + t) % 3 - 1), 0.1, 0.0, 0.05])
        else:
            rows.append([0.1 * ((i + t) % 7 - 3), 0.1 * ((3 * i + t) % 5 - 2), 0.05 * ((i + 2 * t) % 3), 0.01 * (i % 100)])

    for i in range(n):
        if (7 * i + 3 * t) % 8 == 0:
            add(i, (i // 8 + t) % 4)
    if idx:
        add(idx[0], (idx[0] + t + 1) % 4)
    return np.array(idx, dtype=np.int32), np.array(modes, dtype=np.int32), np.array(rows, dtype=np.float64)


def test_cpp_node_loop_through_the_facade_equals_blocking_python(tmp_path):
    """tests/cpp/node_loop_async.cpp (rows in, run, positions and sensor rows of a scrambled subset out, two-deep host buffers)
    prints the same facts as the same flight driven through the blocking Python calls."""
    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_RATE_CMD, UavBatch, airframe

    out = json.loads(subprocess.check_output([build(tmp_path, os.path.join(ROOT, "tests", "cpp", "node_loop_async.cpp"))], text=True))
    n, ticks = 256, 40
    i = np.arange(n)
    spawn = np.stack([2.0 * (i % 16), 2.0 * (i // 16), np.full(n, 3.0)], axis=1)
    b = UavBatch([airframe("x500", ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=False)], spawn_xyz=spawn, n=n)
    b.set_collisions(True, False, 100.0)
    sub = np.array([(37 * j + 11) % n for j in range(96)], dtype=np.int32)
    b.set_input(VELOCITY_HDG_RATE_CMD, np.zeros((n, 4)))
    pos_sum, obs_sum, n_rows = 0.0, 0.0, 0
    for t in range(ticks):
        idx, modes, rows = node_commands(t, n)
        n_rows += len(idx)
        set_blocking(b, idx, modes, rows, 4)
        b.run(0.01, 1)
        p = b.get_state(idx=sub, fields=("x",))["x"]
        o = np.concatenate([b.get_odometry(sub), b.get_imu(sub)[:, 3:6], b.get_rangefinder(sub)], axis=1)
        for k in range(len(sub)):
            pos_sum += p[k, 0] + 2.0 * p[k, 1] + 3.0 * p[k, 2]
            obs_sum += o[k, 0] + o[k, 3] + o[k, 6] + o[k, 7] + o[k, 13] + o[k, 16]
    assert out["rows"] == n_rows
    assert out["pos"] == pos_sum and out["obs"] == obs_sum
    assert out["pairs"] == len(b.get_collision_pairs())

"""Snapshots on the GPU (mrsb_snapshot_*): a restored UAV continues exactly as it would have from the moment of the save, bit for
bit, with collisions, on a twin handle from a host image, whatever the bucketing, for any subset and any source record; a save
changes nothing; parameters, gains and handle options are not part of a snapshot."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import rand
from oracle import binding as O
from test_collisions_gpu import ENGINE, geometry, sorted_pairs
from test_respawn import commands, edits, step, type_of, types
from test_respawn_gpu import assert_equal, gpu_dirty, state

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER_BYTES = 48
ROWS = 88
RATE_INTEGRAL_ROWS = [26 + 12 + 9 + c for c in range(3)]  # pid block at 26, integrals at +12, rate PIDs 9..11


def Batch(*a, **kw):
    from mrs_multirotor_simulator_b200 import UavBatch

    return UavBatch(*a, **kw)


def records(img, n):
    """The image's records: rows [88][n] (as uint64 bits), flags [n], modes [n]."""
    a = np.frombuffer(img, dtype=np.uint8, offset=HEADER_BYTES)
    rows = a[:8 * ROWS * n].view(np.uint64).reshape(ROWS, n)
    flags = a[8 * ROWS * n:8 * ROWS * n + 4 * n].view(np.uint32)
    return rows, flags, a[8 * ROWS * n + 4 * n:]


def image(b):
    s = b.snapshot()
    s.save()
    out = s.to_bytes()
    s.free()
    return out


def assert_records_equal(img_a, img_b, n, sel_a=slice(None), sel_b=slice(None), what=""):
    ra, rb = records(img_a, n), records(img_b, n)
    assert np.array_equal(ra[0][:, sel_a], rb[0][:, sel_b]), f"{what}: rows differ"
    assert np.array_equal(ra[1][sel_a], rb[1][sel_b]), f"{what}: flags differ"
    assert np.array_equal(ra[2][sel_a], rb[2][sel_b]), f"{what}: modes differ"


def dense_spawn(n, seed=21, side=50.0):
    return np.stack([rand(seed, 0, n, 0, side), rand(seed, 1, n, 0, side), rand(seed, 2, n, 0, 2)], axis=1), rand(seed, 3, n, -3, 3)


def rich(n, xyz, hdg, crash=None):
    """The airframes of test_respawn on a ground plane, made dirty in every way a snapshot has to carry (gpu_dirty: every mode
    family, feed-forwards, crashes, external forces and moments, a v_prev from set_state, tracker commands, timed-out inputs)
    with iterate_without_input off, and collisions with neighbour lists in the given crash mode (None: collisions off)."""
    b = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz, spawn_heading=hdg, n=n)
    b.set_iterate_without_input(False)
    if crash is not None:
        b.set_collisions(True, crash, 100.0)
        b.set_pair_capacity(16 * n)
    gpu_dirty(b, n, xyz)
    return b


def twin_of(n, xyz, hdg, crash=None):
    """A fresh handle from the same create info with the same parameter edits and handle options as rich() (what a snapshot does
    not hold)."""
    c = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz, spawn_heading=hdg, n=n)
    c.set_iterate_without_input(False)
    if crash is not None:
        c.set_collisions(True, crash, 100.0)
        c.set_pair_capacity(16 * n)
    edits(c, n)
    return c


def leg(b, ticks, by_run):
    pairs = []
    for _ in range(ticks):
        if by_run:
            b.run(0.01, 1)
        else:
            b.make_step(0.01)
            b.handle_collisions()
        pairs.append(b.get_collision_pairs())
    return pairs


@pytest.mark.parametrize("crash", [False, True])
def test_round_trip_is_bit_exact_with_collisions(crash):
    n = 3000
    xyz, hdg = dense_spawn(n)
    b = rich(n, xyz, hdg, crash)
    assert b.collision_info()["neighbour_lists"]
    b.run(0.01, 300)
    s = b.snapshot()
    s.save()
    first = leg(b, 200, by_run=True)
    end_a = image(b)
    s.restore()
    second = leg(b, 200, by_run=False)
    end_b = image(b)
    assert sum(len(p) for p in first) > 0
    for t, (p, q) in enumerate(zip(first, second)):
        assert np.array_equal(p, q), f"pairs of tick {t}"
    assert end_a == end_b
    flags = records(end_a, n)[1]
    assert len(np.unique(records(end_a, n)[2])) == 10 and ((flags & 256) == 0).any()  # every mode; timed-out UAVs wait, frozen


def test_image_resumes_on_a_twin_handle():
    n = 3000
    xyz, hdg = dense_spawn(n, 22)
    a = rich(n, xyz, hdg, False)
    a.run(0.01, 300)
    img = image(a)
    ref = leg(a, 100, by_run=True)
    c = twin_of(n, xyz, hdg, False)
    s = c.snapshot()
    s.load_bytes(img)
    s.restore()
    assert image(c) == img
    got = leg(c, 100, by_run=True)
    assert sum(len(p) for p in ref) > 0
    for t, (p, q) in enumerate(zip(ref, got)):
        assert np.array_equal(p, q), f"pairs of tick {t}"
    assert image(a) == image(c)


def test_bucketing_changes_no_bit(monkeypatch):
    n = 3 * 58001
    xyz, hdg = dense_spawn(n, 23, side=400.0)
    a = rich(n, xyz, hdg)
    monkeypatch.setenv("MRSB_NO_BUCKETS", "1")
    b = rich(n, xyz, hdg)
    monkeypatch.delenv("MRSB_NO_BUCKETS")
    img_a, img_b = image(a), image(b)
    assert img_a == img_b
    step(a, 30)
    step(b, 30)
    sa, sb = a.snapshot(), b.snapshot()
    sa.load_bytes(img_b)  # each takes the other's image
    sb.load_bytes(img_a)
    sa.restore()
    sb.restore_device()
    assert image(a) == img_a and image(b) == img_a
    step(a, 50)
    step(b, 50)
    assert image(a) == image(b)


def test_partial_restore_host_and_device_forms():
    import torch

    n = 3 * 2000 + 7
    xyz, hdg = dense_spawn(n, 24, side=200.0)
    hs = [rich(n, xyz, hdg) for _ in range(4)]  # a: host form, b: device form, c: no restore, d: restores everybody
    snaps = [h.snapshot() for h in hs]
    for s in snaps:
        s.save()
    for h in hs:
        step(h, 50)
    sub = np.flatnonzero(O.u01(31, 0, np.arange(n)) < 0.3).astype(np.int32)
    rest = np.setdiff1d(np.arange(n), sub).astype(np.int32)
    src = np.full(n, -1, dtype=np.int32)
    src[sub] = sub
    src[rest[::2]] = n + 7  # out of range: untouched
    src_dev = torch.as_tensor(src, device="cuda:0")
    torch.cuda.synchronize()
    snaps[0].restore(idx=sub)
    snaps[1].restore_device(src_dev.data_ptr())
    snaps[3].restore()
    hs[1].sync()
    assert image(hs[0]) == image(hs[1])
    for h in hs:
        commands(h, n, 5, xyz)
        step(h, 100)
    img = [image(h) for h in hs]
    assert img[0] == img[1]
    assert_records_equal(img[0], img[3], n, sub, sub, "restored UAVs")
    assert_records_equal(img[0], img[2], n, rest, rest, "UAVs not restored")
    assert_equal(state(hs[0], sub), state(hs[3], sub), "restored UAVs")
    assert_equal(state(hs[1], rest), state(hs[2], rest), "UAVs not restored")
    assert not np.array_equal(records(img[0], n)[0][:, sub], records(img[2], n)[0][:, sub])


@pytest.mark.parametrize("form", ["host", "device"])
def test_permuted_source_follows_the_source_uav(form):
    import torch

    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_CMD, airframe

    n = 58001
    x500 = airframe("x500", ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=True)
    xyz = np.stack([4.0 * (np.arange(n) % 256), 4.0 * (np.arange(n) // 256), np.zeros(n)], axis=1)
    cmd = np.stack([rand(4, 0, n, -1, 1), rand(4, 1, n, -1, 1), rand(4, 2, n, 0.2, 1.5), rand(4, 3, n, -3, 3)], axis=1)
    a, b = (Batch([x500], spawn_xyz=xyz, n=n) for _ in range(2))
    for h in (a, b):
        h.set_input(VELOCITY_HDG_CMD, cmd)
        for _ in range(20):
            h.make_step(0.01, 10)
    s = b.snapshot()
    s.save()
    for _ in range(5):
        b.make_step(0.01, 10)
    perm = np.random.default_rng(5).permutation(n).astype(np.int32)
    if form == "host":
        s.restore(src=perm)
    else:
        p = torch.as_tensor(perm, device="cuda:0")
        torch.cuda.synchronize()
        s.restore_device(p.data_ptr())
        b.sync()
    for h in (a, b):
        for _ in range(10):
            h.make_step(0.01, 10)
    assert b.step_info()["variant"] == "staged"  # the batch kept its one mode
    ra, rb = state(a), state(b)
    for k in ra:
        assert np.array_equal(rb[k], ra[k][perm]), k


def test_parameters_and_gains_are_kept():
    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_CMD

    n = 600
    xyz, hdg = dense_spawn(n, 25, side=100.0)
    b = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz, spawn_heading=hdg, n=n)
    commands(b, n, 3, xyz)
    step(b, 50)
    assert b.get_controller_params(0).rate_ki == 0.0
    s = b.snapshot()
    s.save()
    step(b, 20)
    m = np.arange(0, n, 3, dtype=np.int32)
    b.set_mass(2.5, idx=m)
    g = np.arange(1, n, 3, dtype=np.int32)
    b.set_controller_params("rate", [5.0, 0.05, 0.3], idx=g)
    b.set_controller_params("velocity", [2.5, 0.06, 0.02, 4.5], idx=g)
    before = {i: (bytes(b.get_params(i)), bytes(b.get_controller_params(i))) for i in range(0, n, 7)}
    step(b, 20)  # the rate integrals of g become non-zero
    assert np.any(records(image(b), n)[0][RATE_INTEGRAL_ROWS][:, g] != 0)
    s.restore()
    for i, (p, c) in before.items():
        assert bytes(b.get_controller_params(i)) == c
        got = b.get_params(i)
        ref = type(got).from_buffer_copy(p)
        ref.takeoff_patch_enabled = got.takeoff_patch_enabled  # the live flag is part of the record
        assert bytes(got) == bytes(ref)
    assert b.get_params(0).mass == 2.5 and b.get_controller_params(1).rate_ki == 0.3
    assert not np.any(records(image(b), n)[0][RATE_INTEGRAL_ROWS])  # saved with ki == 0: zero

    from mrs_multirotor_simulator_b200 import airframe

    u = 58001
    import torch

    c = Batch([airframe("x500")], spawn_xyz=np.stack([4.0 * (np.arange(u) % 256), 4.0 * (np.arange(u) // 256), np.full(u, 2.0)], axis=1), n=u)
    cmd = torch.zeros((u, 4), dtype=torch.float64, device="cuda:0")
    torch.cuda.synchronize()
    c.set_input_device(VELOCITY_HDG_CMD, cmd.data_ptr(), 4)
    c.make_step(0.01, 10)
    sc = c.snapshot()
    sc.save()
    c.set_input(1, np.full((1, 8), 0.5), idx=[7])  # a second mode: the batch is mixed
    c.make_step(0.01, 10)
    assert c.step_info()["variant"] == "direct"
    sc.restore()  # everybody its own record: the saved mode again
    c.make_step(0.01, 10)
    assert c.step_info()["variant"] == "staged"
    c.set_input(1, np.full((1, 8), 0.5), idx=[7])
    sc.restore_device()
    c.set_input_device(VELOCITY_HDG_CMD, cmd.data_ptr(), 4)
    c.make_step(0.01, 10)
    assert c.step_info()["variant"] == "staged"
    c.sync()


@pytest.mark.parametrize("form", ["host", "device"])
def test_restored_forces_are_replaced_by_the_next_pass(form):
    import torch

    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_CMD, airframe

    n = 1600
    types_ = [airframe("x500"), airframe("f550")]
    tou = (np.arange(n) % 2).astype(np.int32)
    k = np.arange(n)
    xyz = np.stack([5.0 * (k % 40), 5.0 * (k // 40), np.full(n, 20.0)], axis=1)
    close = np.arange(0, n, 8)
    xyz[close + 1] = xyz[close] + np.array([0.6, 0.2, 0.0])  # pairs
    b = Batch(types_, type_of_uav=tou, spawn_xyz=xyz, n=n)
    b.set_collisions(True, False, 100.0)
    b.set_input(VELOCITY_HDG_CMD, np.zeros((n, 4)))
    b.run(0.01, 3)
    f = b.get_force()
    pushed = close[np.linalg.norm(f[close], axis=1) > 0]
    assert len(pushed) > 50
    s = b.snapshot()
    s.save()
    far = np.stack([1000.0 + 4.0 * np.arange(len(pushed)), np.full(len(pushed), -300.0), np.full(len(pushed), 20.0)], axis=1)
    b.respawn(far, np.zeros(len(pushed)), idx=(pushed + 1).astype(np.int32))  # the partners leave
    b.set_input(VELOCITY_HDG_CMD, np.zeros((n, 4)))
    b.run(0.01, 30)
    info = b.collision_info()
    if form == "host":
        s.restore(idx=pushed.astype(np.int32))
    else:
        src = torch.full((n,), -1, dtype=torch.int32, device="cuda:0")
        src[torch.as_tensor(pushed, device="cuda:0")] = torch.as_tensor(pushed.astype(np.int32), device="cuda:0")
        torch.cuda.synchronize()
        s.restore_device(src.data_ptr())
        b.sync()
    assert np.all(np.linalg.norm(b.get_force(pushed), axis=1) > 0)  # restored non-zero, and nobody near them now
    b.make_step(0.01)
    x = b.get_state()["x"]
    b.handle_collisions()
    arm, prop, mass = geometry(types_, tou)
    ref_pairs, ref_forces, _ = O.collide_snapshot(x, arm, prop, mass, False, 100.0, engine=ENGINE)
    assert np.array_equal(sorted_pairs(ref_pairs), b.get_collision_pairs())
    assert not np.isin(pushed, ref_pairs).any()
    got = b.get_force()
    assert np.all(got[pushed] == 0.0)
    assert np.allclose(ref_forces, got, rtol=1e-12, atol=0)
    assert b.collision_info()["rebuilds"] == info["rebuilds"] + 1


def test_save_is_invisible():
    n = 3000
    xyz, hdg = dense_spawn(n, 26)
    a, b = rich(n, xyz, hdg, False), rich(n, xyz, hdg, False)
    s = b.snapshot()
    for t in range(300):
        a.run(0.01, 1)
        b.run(0.01, 1)
        s.save()
        if t % 50 == 49:
            assert np.array_equal(a.get_collision_pairs(), b.get_collision_pairs()), t
    assert image(a) == image(b) == s.to_bytes()
    ca, cb = a.counters(), b.counters()
    assert ca["launches"] + 300 == cb["launches"]
    ca.pop("launches"), cb.pop("launches")
    assert ca == cb and a.collision_info() == b.collision_info()


def test_sharded_on_one_gpu_with_a_restore_next_to_the_other_shard():
    from test_sharded_gpu import exchange, make_shards

    from mrs_multirotor_simulator_b200 import airframe

    n = 4096
    types_ = [airframe("x500"), airframe("naki"), airframe("t650")]
    tou = (np.arange(n) * 5 % 3).astype(np.int32)
    xyz = np.stack([rand(11, 0, n, 0, 60), rand(11, 1, n, 0, 60), rand(11, 2, n, 2, 8)], axis=1)
    cmd = np.stack([rand(12, 1, n, -1, 1), rand(12, 2, n, -1, 1), rand(12, 3, n, -0.3, 0.3), rand(12, 4, n, -1, 1)], axis=1)
    whole = Batch(types_, type_of_uav=tou, spawn_xyz=xyz, n=n)
    shards = make_shards(types_, tou, xyz, (0, 1500, n))
    for h in [whole] + shards:
        h.set_pair_capacity(8 * n)
        h.set_collisions(True, False, 100.0)
    whole.set_input(O.VELOCITY_HDG_RATE_CMD, cmd)
    for sh in shards:
        sh.set_input(O.VELOCITY_HDG_RATE_CMD, cmd[sh.shard_begin:sh.shard_begin + sh.n])
    glob = np.arange(1600, 1700, dtype=np.int32)  # all on shard 1
    loc = glob - shards[1].shard_begin
    partners = glob - 1000  # all on shard 0
    sw, s0, s1 = whole.snapshot(), shards[0].snapshot(), shards[1].snapshot()
    met = 0
    for t in range(40):
        if t == 3:  # next to UAVs of shard 0
            whole.respawn(xyz[partners] + np.array([0.4, 0.3, 0.2]), np.zeros(len(glob)), idx=glob)
            shards[1].respawn(xyz[partners] + np.array([0.4, 0.3, 0.2]), np.zeros(len(glob)), idx=loc)
            whole.set_input(O.VELOCITY_HDG_RATE_CMD, cmd[glob], idx=glob)
            shards[1].set_input(O.VELOCITY_HDG_RATE_CMD, cmd[glob], idx=loc)
            for s in (sw, s0, s1):
                s.save()
        if t == 10:  # far away
            far = np.stack([500.0 + 4.0 * np.arange(len(glob)), np.full(len(glob), -200.0), np.full(len(glob), 5.0)], axis=1)
            whole.respawn(far, np.zeros(len(glob)), idx=glob)
            shards[1].respawn(far, np.zeros(len(glob)), idx=loc)
        if t == 20:  # both back where they were saved, next to each other across the shard boundary
            import torch

            sw.restore(idx=np.concatenate([glob, partners]))
            s1.restore(idx=loc)
            src = torch.full((shards[0].n,), -1, dtype=torch.int32, device="cuda:0")
            src[torch.as_tensor(partners, device="cuda:0")] = torch.as_tensor(partners, device="cuda:0")
            torch.cuda.synchronize()
            s0.restore_device(src.data_ptr())
            shards[0].sync()
        whole.make_step(0.01)
        whole.handle_collisions()
        for sh in shards:
            sh.make_step(0.01)
            sh.publish_positions()
        exchange(shards)
        for sh in shards:
            sh.handle_collisions_gathered()
        pairs = np.concatenate([sh.get_collision_pairs() for sh in shards])
        assert np.array_equal(whole.get_collision_pairs(), sorted_pairs(pairs)), t
        if t == 20:
            met = np.isin(pairs[:, 0], glob).sum()
    assert met > 0  # the restored UAVs met shard 0's restored ones
    ref = state(whole)
    got = [state(sh) for sh in shards]
    for k in ref:
        assert np.array_equal(ref[k], np.concatenate([g[k] for g in got])), k


def test_pull_exchange_sees_a_restore_next_to_a_peer():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29543", os.path.join(ROOT, "tests", "snapshot_multi_gpu_check.py")], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "SNAPSHOT_MULTI_GPU_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_invalid_arguments_and_empty_calls():
    import ctypes as C

    import torch

    from mrs_multirotor_simulator_b200._lib import MrsbError

    n = 256
    xyz, hdg = dense_spawn(n, 27)
    b = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz, spawn_heading=hdg, n=n)
    commands(b, n, 3, xyz)
    step(b, 10)
    L = b._L
    s = b.snapshot()
    for fn in (s.restore, s.restore_device, s.to_bytes):
        with pytest.raises(MrsbError) as e:
            fn()
        assert e.value.code == -5  # never saved
    s.save()
    before = state(b)
    img = s.to_bytes()
    size = C.c_size_t(0)
    assert L.mrsb_snapshot_image_size(b.h, C.byref(size)) == 0 and size.value == len(img) == HEADER_BYTES + 709 * n
    for idx, src in (([n], None), ([-1], None), ([0, 1], [0, n]), ([0], [-1]), (None, [n + 1])):
        with pytest.raises(MrsbError) as e:
            s.restore(idx=idx, src=src)
        assert e.value.code == -1
    assert L.mrsb_snapshot_restore(b.h, s.id, n + 1, None, None) == -1
    assert L.mrsb_snapshot_restore(b.h, s.id, 0, None, None) == 0
    for bad in (img[:-1], img + b"\0", b"X" + img[1:]):
        with pytest.raises(MrsbError) as e:
            s.load_bytes(bad)
        assert e.value.code == -1
    other = Batch(types(), type_of_uav=type_of(n + 1), spawn_xyz=dense_spawn(n + 1, 27)[0], n=n + 1)
    so = other.snapshot()
    so.save()
    wrong_n = bytearray(so.to_bytes()[:len(img)])
    with pytest.raises(MrsbError) as e:
        s.load_bytes(bytes(wrong_n))  # right size, n_local of another shard
    assert e.value.code == -1
    for sid in (s.id + 100, -3):
        assert L.mrsb_snapshot_save(b.h, sid) == -1
        assert L.mrsb_snapshot_restore(b.h, sid, 1, None, None) == -1
        assert L.mrsb_snapshot_restore_device(b.h, sid, None) == -1
        assert L.mrsb_snapshot_free(b.h, sid) == -1
    assert L.mrsb_snapshot_create(b.h, None) == -1
    assert L.mrsb_snapshot_save(None, s.id) == -1
    assert_equal(before, state(b), "after failed and empty calls")
    step(b, 10)
    moved = state(b)
    src = torch.full((n,), n, dtype=torch.int32, device="cuda:0")
    src[5] = 9
    src[6] = -1
    torch.cuda.synchronize()
    s.restore_device(src.data_ptr())
    b.sync()
    ref = records(img, n)
    now = records(image(b), n)
    assert np.array_equal(now[0][:, 5], ref[0][:, 9]) and now[1][5] == ref[1][9] and now[2][5] == ref[2][9]
    after = state(b)
    keep = np.setdiff1d(np.arange(n), [5])
    for k in after:
        assert np.array_equal(after[k][keep], moved[k][keep]), k
    dead = s.id
    s.free()
    assert L.mrsb_snapshot_save(b.h, dead) == -1 and L.mrsb_snapshot_free(b.h, dead) == -1
    s2 = b.snapshot()
    assert s2.id != dead
    other.close()
    b.close()  # frees s2 with the handle


def checksum(b):
    st = b.get_state()
    s = 0.0
    for k in range(b.n):  # in order, like the C++ program
        s += st["x"][k, 0] + 2.0 * st["x"][k, 1] + 3.0 * st["x"][k, 2] + st["v"][k, 2]
    return s


def test_snapshot_loop_through_the_facade_equals_the_python_mirror(tmp_path):
    from test_cpp_facade import build

    from mrs_multirotor_simulator_b200 import POSITION_CMD, airframe

    out = json.loads(subprocess.check_output([build(tmp_path, os.path.join(ROOT, "tests", "cpp", "snapshot_loop.cpp"))], text=True))
    n = 512
    i = np.arange(n)
    spawn_ = np.stack([1.5 * (i % 32), 1.5 * (i // 32), np.zeros(n)], axis=1)
    x500 = airframe("x500", ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=True)
    b = Batch([x500], spawn_xyz=spawn_, spawn_heading=0.01 * i, n=n)
    b.set_collisions(True, False, 100.0)
    cmd = np.stack([spawn_[:, 0] + 0.5 * (i % 5), spawn_[:, 1] - 0.25 * (i % 3), 2.0 + 0.1 * (i % 7), np.full(n, 0.3)], axis=1)
    for k in range(n):  # one setInput per UAV, like the C++ program
        b.set_input(POSITION_CMD, cmd[k:k + 1], idx=[k])
    b.run(0.01, 100)
    s = b.snapshot()
    s.save()
    sums = []
    for branch in range(3):
        if branch == 1:
            s.restore()
        if branch == 2:
            s.restore(src=(i + 34) % n)
        b.run(0.01, 50)
        sums.append(checksum(b))
    img = s.to_bytes()
    c = Batch([x500], spawn_xyz=spawn_, spawn_heading=0.01 * i, n=n)
    c.set_collisions(True, False, 100.0)
    sc = c.snapshot()
    sc.load_bytes(img)
    sc.restore()
    c.run(0.01, 50)
    assert sums[0] == sums[1] == checksum(c)
    assert out == {"sums": sums, "resumed": sums[0], "image_bytes": len(img), "pairs": len(b.get_collision_pairs())}

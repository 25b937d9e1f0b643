"""Episode reset on the GPU (mrsb_respawn, mrsb_respawn_masked_device): a respawned UAV is a freshly created one with the same
parameters and gains, bit for bit; the masked device form equals the host form; the collision pass, the tick graph, the staged
kernel and sharded runs stay right around it."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import TOL, assert_parity, rand
from oracle import binding as O
from test_collisions_gpu import ENGINE, geometry, sorted_pairs
from test_respawn import RespawnOracle, commands, dirty, fresh_like, spawn, step, type_of, types

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("x", "v", "R", "omega", "motor_rpm", "v_prev", "imu")


def Batch(*a, **kw):
    from mrs_multirotor_simulator_b200 import UavBatch

    return UavBatch(*a, **kw)


def gpu_dirty(b, n, xyz):
    """dirty() plus what only the library has: set_state with a v_prev override, a tracker command, an input timeout."""
    dirty(b, n, xyz)
    s = np.arange(4, n, 11, dtype=np.int32)
    b.set_state(idx=s, v=np.tile([0.3, -0.2, 0.1], (len(s), 1)))
    t = np.arange(5, n, 13, dtype=np.int32)
    b.set_tracker_cmd(np.tile([0.2, 0.1, 0.3, 0.05, -0.05, 0.1, 0.2, 1, 1, 1, 1], (len(t), 1)), idx=t)
    b.timeout_input(idx=np.arange(6, n, 17, dtype=np.int32))
    step(b, 20)


def state(b, idx=None, sample=()):
    st = b.get_full_state(idx)
    out = {k: st[k] for k in FIELDS}
    out["crashed"] = b.has_crashed(idx)
    out["force"] = b.get_force(idx)
    out["mode"] = b.get_input_mode(idx)
    for i in sample:
        out[f"params{i}"] = np.frombuffer(bytes(b.get_params(int(i))), dtype=np.uint8)
        out[f"gains{i}"] = np.frombuffer(bytes(b.get_controller_params(int(i))), dtype=np.uint8)
    return out


def assert_equal(a, b, what):
    bad = [k for k in a if not np.array_equal(a[k], b[k])]
    assert not bad, f"{what}: {bad} differ"


def respawn_poses(n, seed=2):
    xyz, hdg = spawn(n, seed)
    xyz[::2, 2] = 0.0  # on the ground: the take-off patch engages again
    xyz[1::2, 2] = 5.0
    return xyz, hdg


def test_respawn_equals_a_fresh_handle_bit_for_bit():
    """Bucketed 4/6/8-motor batch (3 x 58,001): respawned UAVs equal a handle created at the respawn poses with the same edits and
    gains; the UAVs not respawned equal a handle that ran the same sequence without the respawn."""
    n = 3 * 58001
    xyz0, hdg0 = spawn(n, 1)
    xyz, hdg = respawn_poses(n)
    a = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    c = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    for h in (a, c):
        gpu_dirty(h, n, xyz0)
    sub = np.flatnonzero(np.arange(n) % 4 < 2).astype(np.int32)  # all airframes, crashed, mass-edited and custom-gain UAVs
    before = a.has_crashed(sub)
    assert before.sum() > 1000 and (a.get_input_mode(sub) != 0).all()
    a.respawn(xyz[sub], hdg[sub], idx=sub)
    b = fresh_like(Batch, n, xyz, hdg)
    b.set_external_moment(np.zeros((1, 3)), idx=[0])  # the moment-enabled stepping variant, like a and c
    sample = [int(i) for i in sub[:: len(sub) // 40]]
    assert_equal(state(a, sub, sample), state(b, sub, sample), "right after the respawn")
    assert (a.get_input_mode(sub) == 0).all() and not a.has_crashed(sub).any()
    assert all(a.get_params(int(i)).takeoff_patch_enabled for i in sample)
    rest = np.setdiff1d(np.arange(n), sub).astype(np.int32)
    for h in (a, b, c):
        commands(h, n, 5, xyz)
        step(h, 500)
    assert_equal(state(a, sub, sample), state(b, sub, sample), "5 s after the respawn")
    assert_equal(state(a, rest), state(c, rest), "UAVs not respawned")
    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_CMD

    cmd = np.stack([rand(6, 0, n, -1, 1), rand(6, 1, n, -1, 1), rand(6, 2, n, -0.5, 1), rand(6, 3, n, -3, 3)], axis=1)
    for h in (a, b, c):
        h.set_input(VELOCITY_HDG_CMD, cmd)  # one mode for the whole batch
        for _ in range(50):
            h.make_step(0.01, 10)
    assert_equal(state(a, sub, sample), state(b, sub, sample), "10 s after the respawn")
    assert_equal(state(a, rest), state(c, rest), "UAVs not respawned, 10 s")
    consumed = [i for i in sample if i % 2 == 0]  # respawned on the ground, then took off again
    assert consumed and not all(a.get_params(i).takeoff_patch_enabled for i in consumed)


def test_respawn_against_the_oracle_in_every_mode_family():
    n = 90
    xyz0, hdg0 = spawn(n, 1)
    xyz, hdg = respawn_poses(n)
    orc = RespawnOracle(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    gpu = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    for s in (orc, gpu):
        dirty(s, n, xyz0)
    sub = np.arange(0, n, 2, dtype=np.int32)
    sub = np.union1d(sub, np.arange(2, n, 7)).astype(np.int32)  # every crashed UAV too
    for s in (orc, gpu):
        s.respawn(xyz[sub], hdg[sub], idx=sub)
    assert_parity(orc, gpu, what="right after the respawn")
    for s in (orc, gpu):
        commands(s, n, 5, xyz)
    on_ground = [int(i) for i in sub if xyz[i, 2] == 0.0]
    assert all(gpu.get_params(i).takeoff_patch_enabled for i in on_ground)
    for t in range(10):  # 10 s
        orc.make_step(0.01, 100)
        step(gpu, 100)
        assert_parity(orc, gpu, what=f"{t + 1} s after the respawn")
        assert np.array_equal(orc.has_crashed(), gpu.has_crashed())
    flags = [gpu.get_params(i).takeoff_patch_enabled for i in on_ground]
    assert flags == [orc.get_params(i).takeoff_patch_enabled for i in on_ground]
    assert not all(flags)  # the patch engaged again and was consumed at lift-off


def _torch_args(xyz, hdg, mask):
    import torch

    dev = torch.device("cuda:0")
    m = torch.as_tensor(mask, dtype=torch.bool, device=dev)
    x = torch.as_tensor(np.ascontiguousarray(xyz), dtype=torch.float64, device=dev)
    h = torch.as_tensor(np.ascontiguousarray(hdg), dtype=torch.float64, device=dev)
    return m, x, h


def masked(b, xyz, hdg, mask):
    import torch

    m, x, h = _torch_args(xyz, hdg, mask)
    torch.cuda.synchronize()
    b.respawn_masked_device(m.data_ptr(), x.data_ptr(), h.data_ptr())
    b.sync()  # keeps the tensors alive until the kernel has read them


def test_masked_device_form_equals_host_form():
    n = 3 * 2000 + 7
    xyz0, hdg0 = spawn(n, 1)
    xyz, hdg = respawn_poses(n, 3)
    d = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    e = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    for h in (d, e):
        gpu_dirty(h, n, xyz0)
    mask = O.u01(9, 0, np.arange(n)) < 0.3
    mask[2::7] = True  # crashed ones
    sub = np.flatnonzero(mask).astype(np.int32)
    d.respawn(xyz[sub], hdg[sub], idx=sub)
    junk = np.where(mask[:, None], xyz, np.nan)  # rows where the mask is clear are not read
    masked(e, junk, np.where(mask, hdg, np.nan), mask)
    sample = [int(i) for i in sub[::50]]
    assert_equal(state(d, None, sample), state(e, None, sample), "after the respawn")
    for h in (d, e):
        commands(h, n, 5, xyz)
        step(h, 200)
    assert_equal(state(d, None, sample), state(e, None, sample), "2 s later")


def _ground_swarm(n):
    """UAVs sitting on the ground 0.7 m apart: pairs in every pass, no force (rebounce 0), no motion: the neighbour lists never
    need a rebuild of their own."""
    from mrs_multirotor_simulator_b200 import airframe

    side = int(np.ceil(np.sqrt(n)))
    k = np.arange(n)
    xyz = np.stack([0.7 * (k % side), 0.7 * (k // side), np.zeros(n)], axis=1)
    b = Batch([airframe("x500", ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=False)], spawn_xyz=xyz, n=n)
    b.set_collisions(True, False, 0.0)
    return b, xyz


def _hover_all(b, n):
    import torch

    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_CMD

    cmd = torch.zeros((n, 4), dtype=torch.float64, device="cuda:0")
    torch.cuda.synchronize()
    b.set_input_device(VELOCITY_HDG_CMD, cmd.data_ptr(), 4)
    b.sync()


def test_empty_mask_changes_nothing_and_one_uav_costs_one_rebuild():
    n = 4096
    runs = {}
    for variant in ("none", "empty", "one"):
        b, xyz = _ground_swarm(n)
        _hover_all(b, n)
        b.run(0.01, 20)
        mask = np.zeros(n, dtype=bool)
        if variant == "one":
            mask[77] = True
        if variant != "none":
            masked(b, xyz, np.zeros(n), mask)
        _hover_all(b, n)  # the RL order: respawn -> commands for the whole batch -> step
        b.run(0.01, 40)
        runs[variant] = (state(b), b.get_collision_pairs(), b.collision_info(), b.step_info())
    assert runs["none"][2]["passes"] == 60
    assert_equal(runs["none"][0], runs["empty"][0], "all-zero mask")
    assert np.array_equal(runs["none"][1], runs["empty"][1]) and len(runs["none"][1]) > 0
    assert runs["none"][2] == runs["empty"][2]
    assert runs["one"][2]["rebuilds"] == runs["none"][2]["rebuilds"] + 1, (runs["one"][2], runs["none"][2])
    assert runs["one"][3] == runs["none"][3]  # the same stepping kernel: the batch is one mode again after the commands


@pytest.mark.parametrize("crash", [False, True])
def test_collisions_with_neighbour_lists_around_respawns(crash):
    from mrs_multirotor_simulator_b200 import airframe

    n = 1600
    types_ = [airframe("x500"), airframe("f550")]
    tou = (np.arange(n) % 2).astype(np.int32)
    side = 40
    k = np.arange(n)
    xyz0 = np.stack([5.0 * (k % side), 5.0 * (k // side), np.full(n, 20.0)], axis=1)
    b = Batch(types_, type_of_uav=tou, spawn_xyz=xyz0, n=n)
    assert b.collision_info()["neighbour_lists"]
    b.set_collisions(True, crash, 100.0)
    b.set_input(O.VELOCITY_HDG_RATE_CMD, np.stack([rand(8, 1, n, -1, 1), rand(8, 2, n, -1, 1), np.zeros(n), np.zeros(n)], axis=1))
    arm, prop, mass = geometry(types_, tou)
    crashed = np.zeros(n, dtype=bool)
    hits = 0
    for t in range(60):
        if t in (10, 30, 45):
            x = b.get_state()["x"]
            into = np.arange(100 + t, 400, 3, dtype=np.int32)  # next to a neighbour: into a cluster
            out = np.flatnonzero(b.has_crashed())[:20].astype(np.int32) if t > 10 else np.arange(0, 30, dtype=np.int32)
            out = np.setdiff1d(out, into).astype(np.int32)
            mask = np.zeros(n, dtype=bool)
            mask[out] = True
            dst = x.copy()
            dst[into] = x[into + 1] + np.array([0.5, 0.2, 0.1])
            dst[out] = np.stack([250.0 + 4.0 * np.arange(len(out)), np.full(len(out), -50.0), np.full(len(out), 30.0)], axis=1)  # away from all
            b.respawn(dst[into], np.zeros(len(into)), idx=into)
            masked(b, dst, np.zeros(n), mask)
            crashed[into] = False
            crashed[out] = False
            b.set_input(O.VELOCITY_HDG_RATE_CMD, np.zeros((n, 4)))
            assert not b.has_crashed(np.concatenate([into, out])).any()
        b.make_step(0.01)
        x = b.get_state()["x"]
        b.handle_collisions()
        ref_pairs, ref_forces, ref_crashed = O.collide_snapshot(x, arm, prop, mass, crash, 100.0, engine=ENGINE)
        assert np.array_equal(sorted_pairs(ref_pairs), b.get_collision_pairs()), t
        if not crash:
            assert np.allclose(ref_forces, b.get_force(), rtol=1e-12, atol=0), t
        crashed |= ref_crashed.astype(bool)
        assert np.array_equal(crashed, b.has_crashed().astype(bool)), t
        hits += len(ref_pairs)
    assert hits > 0
    info = b.collision_info()
    assert info["rebuilds"] < info["passes"], info  # lists were used between the respawns


def test_respawned_uav_waits_for_a_command_without_iterate_without_input():
    n = 300
    xyz0, hdg0 = spawn(n, 1, z=3.0)
    b = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    b.set_iterate_without_input(False)
    commands(b, n, 3, xyz0)
    step(b, 50)
    sub = np.arange(0, n, 3, dtype=np.int32)
    xyz = xyz0[sub] + np.array([0.0, 0.0, 5.0])
    b.respawn(xyz, hdg0[sub], idx=sub)
    frozen = state(b, sub)
    step(b, 50)
    assert_equal(frozen, state(b, sub), "respawned UAVs without a command")
    b.set_input(O.VELOCITY_HDG_CMD, np.tile([0.5, 0.0, 0.3, 0.0], (len(sub), 1)), idx=sub)
    step(b, 50)
    assert np.all(b.get_state(sub)["x"][:, 2] != xyz[:, 2])


def test_c3_loop_with_masked_respawns():
    """BASELINE C3 (65,536 x500, VelocityHdg, K = 10) as an RL loop: about 1 % respawned by mask every 10 launches, each respawn
    followed by the whole batch's commands from the device.  The staged kernel keeps running; a sample of UAVs agrees with the
    oracle; mrsb_run with the respawns between calls equals the same ticks issued one by one."""
    import torch

    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_CMD, airframe

    n, K = 65536, 10
    x500 = airframe("x500", ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=True)
    xyz0, hdg0 = spawn(n, 1, z=0.0)
    xyz0[:, 0] *= 0.5  # 2 m rows
    b = Batch([x500], spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    pick = np.arange(0, n, 32)
    orc = RespawnOracle([x500], spawn_xyz=xyz0[pick], spawn_heading=hdg0[pick], n=len(pick))
    cmd = np.stack([rand(4, 0, n, -1, 1), rand(4, 1, n, -1, 1), rand(4, 2, n, 0.2, 1.5), rand(4, 3, n, -3, 3)], axis=1)
    cmd_dev = torch.as_tensor(cmd, device="cuda:0")
    torch.cuda.synchronize()
    for cycle in range(6):
        if cycle:
            mask = O.u01(50 + cycle, 0, np.arange(n)) < 0.01
            mask[pick[cycle]] = True  # at least one of the oracle's sample
            xyz, hdg = spawn(n, 60 + cycle, z=0.0)
            xyz[:, 0] *= 0.5
            masked(b, xyz, hdg, mask)
            sel = np.flatnonzero(mask[pick]).astype(np.int32)
            orc.respawn(xyz[pick[sel]], hdg[pick[sel]], idx=sel)
        b.set_input_device(VELOCITY_HDG_CMD, cmd_dev.data_ptr(), 4)
        orc.set_input(O.VELOCITY_HDG_CMD, cmd[pick])
        for _ in range(10):
            b.make_step(0.01, K)
            info = b.step_info()
            assert info["variant"] == "staged" and info["mode"] == VELOCITY_HDG_CMD, info
        orc.make_step(0.01, 10 * K, n_threads=8)
    so, sg = orc.get_state(), b.get_full_state(pick)
    for k, t in TOL.items():
        d = float(np.max(np.abs(so[k] - sg[k])))
        assert d <= t, f"{k}: {d:.3e}"

    def tick_loop(one_by_one):
        h = Batch([x500], spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
        h.set_collisions(True, False, 100.0)
        h.set_input_device(VELOCITY_HDG_CMD, cmd_dev.data_ptr(), 4)
        for cycle in range(4):
            if cycle:
                mask = O.u01(70 + cycle, 0, np.arange(n)) < 0.01
                xyz, hdg = spawn(n, 80 + cycle, z=0.0)
                xyz[:, 0] *= 0.5
                masked(h, xyz, hdg, mask)
                h.set_input_device(VELOCITY_HDG_CMD, cmd_dev.data_ptr(), 4)
            if one_by_one:
                for _ in range(10):
                    h.make_step(0.01, K)
                    h.handle_collisions()
            else:
                h.run(0.01, 10, K)
        out = state(h)
        out["pairs"] = h.get_collision_pairs()
        return out, h.collision_info()

    (ra, ia), (rb, ib) = tick_loop(False), tick_loop(True)
    assert_equal(ra, rb, "mrsb_run vs one tick at a time")
    assert len(ra["pairs"]) > 0 and ia["rebuilds"] == ib["rebuilds"] and ia["rebuilds"] >= 4


def test_sharded_on_one_gpu_with_a_respawn_on_one_shard():
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
        h.set_collisions(True, True, 100.0)
    whole.set_input(O.VELOCITY_HDG_RATE_CMD, cmd)
    for sh in shards:
        sh.set_input(O.VELOCITY_HDG_RATE_CMD, cmd[sh.shard_begin:sh.shard_begin + sh.n])
    glob = np.arange(1600, 1700, dtype=np.int32)  # all on shard 1
    dst = xyz[glob - 1000] + np.array([0.4, 0.3, 0.2])  # next to UAVs of shard 0
    for t in range(30):
        if t == 10:
            whole.respawn(dst, np.zeros(len(glob)), idx=glob)
            shards[1].respawn(dst, np.zeros(len(glob)), idx=glob - shards[1].shard_begin)
            whole.set_input(O.VELOCITY_HDG_RATE_CMD, cmd[glob], idx=glob)
            shards[1].set_input(O.VELOCITY_HDG_RATE_CMD, cmd[glob], idx=glob - shards[1].shard_begin)
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
        if t == 10:
            assert np.isin(pairs[:, 0], glob).sum() > 0  # the respawned UAVs met shard 0's
    ref = state(whole)
    got = [state(sh) for sh in shards]
    for k in ref:
        assert np.array_equal(ref[k], np.concatenate([g[k] for g in got])), k


def test_pull_exchange_sees_a_respawn_next_to_a_peer():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29541", os.path.join(ROOT, "tests", "respawn_multi_gpu_check.py")], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "RESPAWN_MULTI_GPU_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_invalid_arguments_and_empty_calls():
    import ctypes as C

    from mrs_multirotor_simulator_b200._lib import MrsbError

    n = 256
    xyz0, hdg0 = spawn(n, 1, z=2.0)
    b = Batch(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    commands(b, n, 3, xyz0)
    step(b, 10)
    before = state(b)
    for idx in ([n], [-1], [0, n + 5]):
        with pytest.raises(MrsbError) as e:
            b.respawn(np.zeros((len(idx), 3)), np.zeros(len(idx)), idx=idx)
        assert e.value.code == -1
    L = b._L
    one = (C.c_int32 * 1)(3)
    xyz = (C.c_double * 3)(1.0, 2.0, 3.0)
    hdg = (C.c_double * 1)(0.0)
    assert L.mrsb_respawn(b.h, 1, one, None, hdg) == -1
    assert L.mrsb_respawn(b.h, 1, one, xyz, None) == -1
    assert L.mrsb_respawn(b.h, n + 1, None, None, None) == -1
    assert L.mrsb_respawn(b.h, 0, None, None, None) == 0
    assert L.mrsb_respawn(b.h, 0, one, xyz, hdg) == 0
    assert L.mrsb_respawn_masked_device(b.h, None, None, None) == -1
    assert L.mrsb_respawn_masked_device(None, None, None, None) == -1
    b.respawn(np.zeros((0, 3)), np.zeros(0), idx=np.zeros(0, dtype=np.int32))
    assert_equal(before, state(b), "after failed and empty calls")


def test_episode_loop_through_the_facade_equals_the_python_mirror(tmp_path):
    from test_cpp_facade import build

    from mrs_multirotor_simulator_b200 import POSITION_CMD, airframe

    out = json.loads(subprocess.check_output([build(tmp_path, os.path.join(ROOT, "tests", "cpp", "episode_loop.cpp"))], text=True))
    n = 512
    i = np.arange(n)
    spawn_ = np.stack([4.0 * (i % 32), 4.0 * (i // 32), np.zeros(n)], axis=1)
    b = Batch([airframe("x500", ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=True)], spawn_xyz=spawn_, spawn_heading=0.01 * i, n=n)
    respawned = 0
    for episode in range(4):
        cmd = np.stack([spawn_[:, 0] + 0.5 * ((i + episode) % 5), spawn_[:, 1] - 0.25 * ((i + episode) % 3), 2.0 + 0.1 * (i % 7),
                        np.full(n, 0.1 * episode)], axis=1)
        for k in range(n):  # one setInput per UAV, like the C++ program
            b.set_input(POSITION_CMD, cmd[k:k + 1], idx=[k])
        if episode == 1:
            b.crash(idx=np.arange(0, n, 9))
        b.run(0.01, 50, 2, with_collisions=False)
        x = b.get_state()["x"]
        done = np.flatnonzero(b.has_crashed().astype(bool) | (x[:, 0] > spawn_[:, 0] + 1.0)).astype(np.int32)
        b.respawn(np.stack([spawn_[done, 0], spawn_[done, 1], np.full(len(done), 0.5 * episode)], axis=1), -0.02 * done, idx=done)
        b.respawn([[1.0, 2.0, 3.0]], [0.5], idx=[1])
        respawned += len(done) + 1
    st = b.get_state()
    s = 0.0
    for k in range(n):
        s += st["x"][k, 0] + 2.0 * st["x"][k, 1] + 3.0 * st["x"][k, 2] + st["v"][k, 2] + st["motor_rpm"][k, 0]
    assert out["sum"] == s and out["respawned"] == respawned and out["crashed"] == int(b.has_crashed().sum())
    assert out["one_x"] == [1.0, 2.0, 3.0] and out["one_rpm0"] == 0.0 and out["one_takeoff"] == 1

#!/usr/bin/env python
"""Run under torchrun on 2 GPUs: with the pull exchange (peer memory), a UAV of rank 0 restored by the device form of
mrsb_snapshot_restore to where it was saved, next to a UAV of rank 1 restored the same way, appears in the very next collision pass on both ranks, and
the sharded run equals the unsharded one on rank 0 bit for bit.

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/snapshot_multi_gpu_check.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import rand  # noqa: E402
from mrs_multirotor_simulator_b200 import VELOCITY_HDG_RATE_CMD, UavBatch, airframe  # noqa: E402
from mrs_multirotor_simulator_b200.sharding import connect, shard_range  # noqa: E402


def main():
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    n = 8000
    types = [airframe("x500"), airframe("f550")]
    tou = (np.arange(n) % 2).astype(np.int32)
    xyz = np.stack([rand(41, 0, n, 0, 400), rand(41, 1, n, 0, 400), rand(41, 2, n, 5, 9)], axis=1)  # sparse: lists live long
    cmd = np.stack([rand(42, 1, n, -1, 1), rand(42, 2, n, -1, 1), rand(42, 3, n, -0.2, 0.2), rand(42, 4, n, -1, 1)], axis=1)
    begin, count = shard_range(n, world, rank)
    sl = slice(begin, begin + count)
    mine = UavBatch(types, type_of_uav=tou, spawn_xyz=xyz[sl], n=count, device=local, n_global=n, shard_begin=begin)
    connect(mine, dist)
    assert mine.exchange_mode() == 2, "needs peer access"
    whole = UavBatch(types, type_of_uav=tou, spawn_xyz=xyz, n=n, device=local) if rank == 0 else None
    for b, c in ((mine, cmd[sl]), (whole, cmd)):
        if b is not None:
            b.set_input(VELOCITY_HDG_RATE_CMD, c)
            b.set_collisions(True, False, 100.0)
            b.set_pair_capacity(8 * n)
    mover, target = 17, n - 5  # a UAV of rank 0, one of rank 1
    snap = mine.snapshot()
    snap_whole = whole.snapshot() if whole is not None else None
    hit = False
    for t in range(60):
        if t == 20:
            # rank 0 respawns `mover` next to where `target` is now (rank 1 tells everybody), and every rank saves right after
            tx = [None]
            if rank == world - 1:
                tx = [mine.get_state([target - begin])["x"][0]]
            dist.broadcast_object_list(tx, src=world - 1)
            dst = np.asarray(tx[0]) + np.array([0.5, 0.3, 0.0])
            if rank == 0:
                mine.respawn(dst[None], [0.0], idx=[mover])
            mine.set_input(VELOCITY_HDG_RATE_CMD, cmd[sl])
            snap.save()
            if whole is not None:
                whole.respawn(dst[None], [0.0], idx=[mover])
                whole.set_input(VELOCITY_HDG_RATE_CMD, cmd)
                snap_whole.save()
        if t == 30 and rank == 0:  # far away
            mine.respawn([[5000.0, 5000.0, 9.0]], [0.0], idx=[mover])
            whole.respawn([[5000.0, 5000.0, 9.0]], [0.0], idx=[mover])
        if t == 40:
            # `mover` and `target` are back where they were saved, next to each other (device form, no host synchronisation, on
            # every rank; ranks between them restore nobody)
            src = torch.full((count,), -1, dtype=torch.int32, device=f"cuda:{local}")
            if rank == 0:
                src[mover] = mover
            if rank == world - 1:
                src[target - begin] = target - begin
            torch.cuda.synchronize()
            snap.restore_device(src.data_ptr())
            mine.sync()
            if whole is not None:
                snap_whole.restore(idx=[mover, target])
        mine.make_step(0.01)
        mine.handle_collisions()
        if whole is not None:
            whole.make_step(0.01)
            whole.handle_collisions()
        p = mine.get_collision_pairs()
        if t == 40:
            pair = (mover, target) if rank == 0 else (target, mover)
            hit = any((p[:, 0] == pair[0]) & (p[:, 1] == pair[1]))
        gathered = [None] * world
        dist.all_gather_object(gathered, p)
        if rank == 0:
            allp = np.concatenate(gathered)
            allp = allp[np.lexsort((allp[:, 1], allp[:, 0]))] if len(allp) else allp
            assert np.array_equal(whole.get_collision_pairs(), allp), f"pair lists differ at tick {t}"
    st = mine.get_full_state()
    st["crashed"] = mine.has_crashed()
    st["force"] = mine.get_force()
    gathered = [None] * world
    dist.all_gather_object(gathered, st)
    if rank == 0:
        ref = whole.get_full_state()
        ref["crashed"] = whole.has_crashed()
        ref["force"] = whole.get_force()
        for k in ref:
            assert np.array_equal(ref[k], np.concatenate([g[k] for g in gathered])), f"{k} differs from the unsharded run"
    info = mine.collision_info()
    assert info["neighbour_lists"] and info["rebuilds"] < info["passes"] // 2, info
    hits = [None] * world
    dist.all_gather_object(hits, hit)
    assert all(hits), f"pair ({mover}, {target}) missing right after the restore: {hits}"
    dist.barrier()
    snap.free()
    mine.close()
    if whole is not None:
        snap_whole.free()
        whole.close()
    dist.barrier()
    if rank == 0:
        print("SNAPSHOT_MULTI_GPU_OK", info)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

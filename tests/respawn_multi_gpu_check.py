#!/usr/bin/env python
"""Run under torchrun on 2 GPUs: with the pull exchange (peer memory), a UAV of rank 0 respawned by mask next to a UAV of rank 1
appears in the very next collision pass on both ranks, and the sharded run equals the unsharded one on rank 0 bit for bit.

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/respawn_multi_gpu_check.py
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
    hit = False
    for t in range(40):
        if t == 20:
            # rank 0 respawns `mover` next to where `target` is now (rank 1 tells everybody)
            tx = [None]
            if rank == world - 1:
                tx = [mine.get_state([target - begin])["x"][0]]
            dist.broadcast_object_list(tx, src=world - 1)
            dst = np.asarray(tx[0]) + np.array([0.5, 0.3, 0.0])
            mask = torch.zeros(count, dtype=torch.bool, device=f"cuda:{local}")
            px = torch.zeros((count, 3), dtype=torch.float64, device=f"cuda:{local}")
            ph = torch.zeros(count, dtype=torch.float64, device=f"cuda:{local}")
            if rank == 0:
                mask[mover] = True
                px[mover] = torch.as_tensor(dst)
            torch.cuda.synchronize()
            mine.respawn_masked_device(mask.data_ptr(), px.data_ptr(), ph.data_ptr())
            mine.set_input(VELOCITY_HDG_RATE_CMD, cmd[sl])
            mine.sync()
            if whole is not None:
                whole.respawn(dst[None], [0.0], idx=[mover])
                whole.set_input(VELOCITY_HDG_RATE_CMD, cmd)
        mine.make_step(0.01)
        mine.handle_collisions()
        if whole is not None:
            whole.make_step(0.01)
            whole.handle_collisions()
        p = mine.get_collision_pairs()
        if t == 20:
            pair = (mover, target) if rank == 0 else (target, mover)
            assert any((p[:, 0] == pair[0]) & (p[:, 1] == pair[1])), f"rank {rank}: pair {pair} missing right after the respawn"
            hit = True
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
    assert hit and info["neighbour_lists"] and info["rebuilds"] < info["passes"] // 2, info
    dist.barrier()
    mine.close()
    if whole is not None:
        whole.close()
    dist.barrier()
    if rank == 0:
        print("RESPAWN_MULTI_GPU_OK", info)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

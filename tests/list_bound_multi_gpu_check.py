#!/usr/bin/env python
"""Run under torchrun on >= 2 GPUs: on the pull exchange the neighbour lists' displacement bound travels through the peer
hand-shake, and every rank must take its peers' word.

Head-on pairs are split across ranks: the MOVING UAV of each pair lives on the last rank, its partner HOVERS on rank 0, so rank 0's
own displacement is near zero and its lists stay correct only through the last rank's word.  On every rank, every pass' rebuild
flag must equal the host reference (list_bound_ref.py) fed with the words of all ranks, each computed from that rank's positions
before and after the launch; pairs, forces, crash flags and the final state equal the unsharded run on rank 0 bit for bit.  A
set_state teleport on one rank only must make every rank rebuild at the next pass.

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/list_bound_multi_gpu_check.py
"""
import math
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import list_bound_ref as R  # noqa: E402
from mrs_multirotor_simulator_b200 import VELOCITY_HDG_RATE_CMD, UavBatch, airframe  # noqa: E402
from mrs_multirotor_simulator_b200.sharding import connect, shard_range  # noqa: E402


def layout(n, world, r_list):
    """Hovering UAVs on a 5 m grid; pairs at y < 0 whose first UAV is an index of rank 0 (hovers) and whose second is an index of
    the last rank (flies at it at 1.5 m/s), at separations straddling r_list and inside it."""
    side = int(np.ceil(np.sqrt(n)))
    k = np.arange(n)
    xyz = np.stack([5.0 * (k % side), 5.0 * (k // side), np.full(n, 10.0)], axis=1)
    vel = np.zeros((n, 4))
    b_last, _ = shard_range(n, world, world - 1)
    seps = [r_list + d for d in (-0.004, -0.001, 0.0, 0.001, 0.004, 0.02)] + [math.sqrt(3.0) + f * (r_list - math.sqrt(3.0)) for f in (0.3, 0.6)]
    pairs = []
    for p, s in enumerate(seps):
        i, j = 7 + 3 * p, b_last + 5 + 3 * p
        y = -10.0 - 12.0 * p
        xyz[i] = [30.0, y, 10.0]
        xyz[j] = [30.0 + s, y, 10.0]
        vel[j] = [-1.5, 0.0, 0.0, 0.0]
        pairs.append((i, j))
    return xyz, vel, pairs


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    os.environ.pop("MRSB_NO_P2P", None)
    big = airframe("x500", arm_length=1.2, prop_radius=0.45)  # contact distance above sqrt(3): nanoflann's ball binds
    n = 600 * world
    probe = UavBatch([big], spawn_xyz=np.zeros((4, 3)), n=4, device=local)
    r_list = probe.collision_info()["list_radius"]
    probe.close()
    xyz, vel, pairs = layout(n, world, r_list)
    begin, count = shard_range(n, world, rank)
    sl = slice(begin, begin + count)
    mine = UavBatch([big], spawn_xyz=xyz[sl], n=count, device=local, n_global=n, shard_begin=begin)
    connect(mine, dist)
    assert mine.exchange_mode() == 2, "needs peer access (the pull exchange carries the displacement words)"
    whole = UavBatch([big], spawn_xyz=xyz, n=n, device=local) if rank == 0 else None
    for b, v in ((mine, vel[sl]), (whole, vel)):
        if b is not None:
            b.set_collisions(True, False, 100.0)
            b.set_pair_capacity(n * 8)
            b.set_input(VELOCITY_HDG_RATE_CMD, v)
    info = mine.collision_info()
    assert info["neighbour_lists"], info
    host = R.HostSide(info["skin"])
    rebuilds = info["rebuilds"]
    x = mine.get_state(fields=("x",))["x"]
    flags, n_pairs = [], 0

    def words():
        got = [None] * world
        dist.all_gather_object(got, host.word())
        return [w for r, w in enumerate(got) if r != rank]

    def collide(tag):
        nonlocal rebuilds, n_pairs
        want = host.collide(peer_bits=words())
        mine.handle_collisions()
        if whole is not None:
            whole.handle_collisions()
        r = mine.collision_info()["rebuilds"]
        got, rebuilds = r - rebuilds, r
        flags.append(bool(got))
        assert got == int(want), f"rank {rank}, {tag}: rebuilt={got}, the reference (swarm-wide bound) says {want}"
        p = mine.get_collision_pairs()
        gathered = [None] * world
        dist.all_gather_object(gathered, p)
        if rank == 0:
            allp = np.concatenate(gathered)
            allp = allp[np.lexsort((allp[:, 1], allp[:, 0]))] if len(allp) else allp
            assert np.array_equal(whole.get_collision_pairs(), allp), f"{tag}: pair lists differ from the unsharded run"
            n_pairs += len(allp)
        return bool(got)

    def step():
        nonlocal x
        mine.make_step(0.01)
        if whole is not None:
            whole.make_step(0.01)
        x1 = mine.get_state(fields=("x",))["x"]
        host.launch(R.disp_bits(x, x1))
        x = x1

    for t in range(150):
        step()
        collide(f"pass {t}")
    # a teleport on the last rank only, then one step: every rank's next pass rebuilds
    far = np.arange(n - 8, n)
    newpos = xyz[far] + np.array([0.3, -0.2, 0.1])
    if rank == world - 1:
        mine.set_state(idx=(far - begin).astype(np.int32), x=newpos)
        host.touch()
        x = mine.get_state(fields=("x",))["x"]
    if whole is not None:
        whole.set_state(idx=far.astype(np.int32), x=newpos)
    step()
    assert collide("teleport on the last rank"), f"rank {rank} kept its lists after a peer's teleport"
    for t in range(40):
        step()
        collide(f"after the teleport, pass {t}")
    st = mine.get_full_state()
    st["force"] = mine.get_force()
    st["crashed"] = mine.has_crashed()
    gathered = [None] * world
    dist.all_gather_object(gathered, (st, flags))
    if rank == 0:
        ref = whole.get_full_state()
        ref["force"] = whole.get_force()
        ref["crashed"] = whole.has_crashed()
        for key in ref:
            got = np.concatenate([g[0][key] for g in gathered])
            assert np.array_equal(ref[key], got, equal_nan=True), f"{key} differs from the unsharded run"
        assert all(g[1] == flags for g in gathered), "ranks disagree on when to rebuild"
        unforced_kept = sum(1 for f in flags[1:] if not f)
        assert n_pairs > 0 and sum(flags) >= 3 and unforced_kept >= 20, (n_pairs, sum(flags), unforced_kept)
        print("LIST_BOUND_MULTI_GPU_OK world=%d passes=%d rebuilds=%d pairs=%d" % (world, len(flags), sum(flags), n_pairs), flush=True)
    dist.barrier()
    mine.close()
    if whole is not None:
        whole.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
